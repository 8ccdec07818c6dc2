// C-ABI layer (include/p2m_b200.h): model handle, workspace planning and the forward / backward
// schedules of Pose2Mesh.forward (lib/models/meshnet.py:80-117 of the reference), expressed as
// sequences of the kernels in kernels_simt.cu / cheb_umma.cu on the caller's stream.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "p2m_internal.h"

namespace p2m {

static thread_local std::string g_error;
static thread_local int64_t g_launches = 0;
void set_error(const std::string& msg) { g_error = msg; }
void count_launch(int n) { g_launches += n; }

struct Layer {
  int level, V, fin, fout;
  int bn, relu;
  int block, pos, block_end;
};

struct Block {
  int first_layer, n_layers;
  int level;
  int has_residual;   // 1 <= b <= nb-2   (meshnet.py:108-115)
  int out_unpool;     // 1 <= b <  nb-2   (meshnet.py:111)
  int in_unpool;      // input of this block is the (virtually) unpooled output of the previous block
  int cin, cout;
  InterpTable interp;  // valid when has_residual
};

}  // namespace p2m

using namespace p2m;

struct p2m_model {
  int device = 0;
  int sm_count = 148;
  int precision = P2M_PREC_FP32_SIMT;
  std::vector<DevLevel> levels;
  std::vector<Layer> layers;
  std::vector<Block> blocks;
  int n_joint = 0, cin = 0, cout = 0;
  int fc_in = 0, fc_out = 0;
  int* kernel_status = nullptr;       // device alias of status_host (what the kernels write)
  volatile int* status_host = nullptr;  // mapped pinned host word: set by a tcgen05 kernel whose mbarrier wait timed out
  long long* trace = nullptr;          // debug (P2M_UMMA_TRACE builds): CTA-0 event log of the tcgen05 conv kernel
  int* out_map = nullptr;        // optional fused output gather (vertex -> slot, -1 = dropped)
  int out_rows = 0;
  float* zero_row = nullptr;     // 128 B of zeros (halo source for the empty slots of ragged tiles)
  int elide_padding = 1;         // tcgen05 conv: isolated padding vertices through a plain GEMM with combined weights;
                                 // 1 = on levels where they are >= 40 % of the rows (measured break-even), 2 = wherever
                                 // the tile families exist, 0 = off (p2m_debug_set_elide_padding)
  int dedup_padding = 1;         // eval: among the isolated rows only one representative per class of identical rows is
                                 // computed (DevLevel::rep_tiles); needs elide_padding == 1 (p2m_debug_set_dedup_padding)
  int dw_swap = 1;               // backward: dW from the basis of the gradient, re-using the backward-data pass's L~dz
                                 // (launch_umma_dw_swapped); 0 = rebuild the basis of the layer input (p2m_debug_set_dw_swap)
  int fuse_head = 1;             // eval: the 128 -> 64 conv's epilogue feeds the 64 -> 3 head directly (no 64-wide tensor)
  int split_t1 = 1;              // tcgen05 conv: T1 = L~x in a separate pass (k_cheb_t1) instead of on-chip halo recompute
  int profiling = 0;             // record a CUDA event pair around every conv layer of the eval forward
  std::vector<cudaEvent_t> ev_beg, ev_end;
  std::vector<void*> owned;  // device allocations to free
};

namespace {

// Every entry point that touches the device makes the model's device current for its own duration only: the
// caller's current device is restored on every exit path (single-process multi-GPU callers, nn.DataParallel
// threads, handles garbage-collected at arbitrary times).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) switched = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (switched && prev >= 0) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// A tcgen05 kernel whose bounded mbarrier wait expired wrote the wait's id into the mapped host status word
// (cheb_umma.cu: mbar_timeout).  Checked without any synchronisation at every entry point (and after the stream
// synchronisation of the *_host entry point): the call fails instead of handing out the results of a kernel
// that fell through its barriers.  The word is cleared once reported.
int check_kernel_status(p2m_model* m, const char* where) {
  if (m->status_host == nullptr) return P2M_OK;
  const int code = *m->status_host;
  if (code == 0) return P2M_OK;
  *m->status_host = 0;
  set_error(std::string(where) + ": a tcgen05 kernel of an earlier call on this handle timed out on mbarrier wait #" +
            std::to_string(code) + " (results of that call are invalid)");
  return P2M_ERR_CUDA;
}

constexpr size_t ALIGN = 256;
inline size_t align_up(size_t x) { return (x + ALIGN - 1) / ALIGN * ALIGN; }

struct Bump {
  char* base;
  size_t off = 0;
  explicit Bump(void* p) : base(static_cast<char*>(p)) {}
  template <class T>
  T* take(size_t n) {
    T* p = reinterpret_cast<T*>(base + off);
    off += align_up(n * sizeof(T));
    return p;
  }
};

template <class T>
int upload(p2m_model* m, const std::vector<T>& h, T** out) {
  T* d = nullptr;
  size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
  P2M_CUDA_OK(cudaMalloc(&d, bytes));
  m->owned.push_back(d);
  if (!h.empty()) P2M_CUDA_OK(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = d;
  return P2M_OK;
}

// F.interpolate(x, size=fout, mode='linear', align_corners=False) along the channel axis
// (meshnet.py:109,114; ATen upsample_linear1d: src = scale*(j+0.5)-0.5 clamped at 0, scale = fin/fout).
int build_interp(p2m_model* m, int fin, int fout, InterpTable* t) {
  t->fin = fin;
  t->fout = fout;
  std::vector<int> i0(fout), i1(fout);
  std::vector<float> lam(fout);
  const float scale = (float)fin / (float)fout;
  for (int j = 0; j < fout; ++j) {
    float src = scale * ((float)j + 0.5f) - 0.5f;
    if (src < 0.f) src = 0.f;
    int a = (int)src;
    if (a > fin - 1) a = fin - 1;
    int b = a + ((a < fin - 1) ? 1 : 0);
    i0[j] = a;
    i1[j] = b;
    lam[j] = src - (float)a;
  }
  std::vector<int> tp(fin + 1, 0), ti;
  std::vector<float> tw;
  for (int i = 0; i < fin; ++i) {
    for (int j = 0; j < fout; ++j) {
      float w = 0.f;
      if (i0[j] == i) w += 1.f - lam[j];
      if (i1[j] == i) w += lam[j];
      if (w != 0.f) {
        ti.push_back(j);
        tw.push_back(w);
      }
    }
    tp[i + 1] = (int)ti.size();
  }
  P2M_TRY(upload(m, i0, &t->i0));
  P2M_TRY(upload(m, i1, &t->i1));
  P2M_TRY(upload(m, lam, &t->lam));
  P2M_TRY(upload(m, tp, &t->t_ptr));
  P2M_TRY(upload(m, ti, &t->t_idx));
  P2M_TRY(upload(m, tw, &t->t_w));
  return P2M_OK;
}

struct Sizes {
  size_t max_act = 0;    // floats: max over layers of rows*fout (and fc in/out, and x)
  size_t max_T = 0;      // floats: max rows*3*fin
  size_t max_U = 0;      // floats: max rows*fin
  size_t max_w = 0;      // floats: max fout*3*fin
  size_t max_wpack = 0;  // bytes: packed fp16 hi/lo weight image of the tcgen05 path
  size_t max_thin = 1;   // floats: scratch of the thin head's backward
  int max_f = 0;
};

Sizes model_sizes(const p2m_model* m, int B) {
  Sizes s;
  for (const Layer& L : m->layers) {
    size_t rows = (size_t)B * L.V;
    s.max_act = std::max(s.max_act, rows * L.fout);
    s.max_act = std::max(s.max_act, rows * L.fin);
    s.max_T = std::max(s.max_T, rows * 3 * L.fin);
    s.max_U = std::max(s.max_U, rows * L.fin);
    s.max_w = std::max(s.max_w, (size_t)L.fout * 3 * L.fin);
    if (umma_conv_supported(m->levels[L.level], L.fin, L.fout))
      s.max_wpack = std::max(s.max_wpack, umma_wpack_bytes(L.fin, L.fout));
    s.max_f = std::max(s.max_f, std::max(L.fin, L.fout));
    if (thin_conv_bwd_supported(L.fin, L.fout)) s.max_thin = std::max(s.max_thin, thin_conv_bwd_scratch_floats(rows, L.fin));
  }
  s.max_act = std::max(s.max_act, (size_t)B * m->fc_out);
  s.max_act = std::max(s.max_act, (size_t)B * m->fc_in);
  return s;
}

// Workspace map shared by forward and backward (deterministic bump order).
struct WsMap {
  float* T;
  float* wp_scratch;
  unsigned char* wpack;   // tcgen05 packed weights (one layer at a time)
  float* scale_scratch;   // [2*max_f] eval folded scale/shift
  double* sums;           // [2*max_f]
  float* rot[3];          // eval: rotating activation buffers
  // training: saved tensors
  std::vector<float*> z, a, mean, invstd, scale, shift, wp;
  float* fc_out = nullptr;
  unsigned char* fc_apack = nullptr;  // operand images of the fc GEMM on tcgen05 (launch_umma_gemm)
  unsigned char* fc_wpack = nullptr;
  size_t bytes = 0;
};

WsMap map_workspace(const p2m_model* m, int B, int training, void* base) {
  WsMap w;
  Sizes s = model_sizes(m, B);
  Bump b(base);
  w.T = b.take<float>(s.max_T);
  w.wp_scratch = b.take<float>(s.max_w);
  w.wpack = b.take<unsigned char>(std::max(s.max_wpack, (size_t)16));
  w.scale_scratch = b.take<float>(2 * (size_t)s.max_f);
  w.sums = b.take<double>(2 * (size_t)s.max_f);
  if (umma_gemm_supported(B, m->fc_out, m->fc_in)) {
    w.fc_apack = b.take<unsigned char>(umma_gemm_apack_bytes(B, m->fc_in));
    w.fc_wpack = b.take<unsigned char>(umma_gemm_wpack_bytes(m->fc_out, m->fc_in));
  }
  const size_t nl = m->layers.size();
  if (!training) {
    for (int i = 0; i < 3; ++i) w.rot[i] = b.take<float>(s.max_act);
  } else {
    w.rot[0] = w.rot[1] = w.rot[2] = nullptr;
    w.z.resize(nl); w.a.resize(nl); w.mean.resize(nl); w.invstd.resize(nl);
    w.scale.resize(nl); w.shift.resize(nl); w.wp.resize(nl);
    for (size_t i = 0; i < nl; ++i) {
      const Layer& L = m->layers[i];
      size_t n = (size_t)B * L.V * L.fout;
      w.wp[i] = b.take<float>((size_t)L.fout * 3 * L.fin);
      if (L.bn) {
        w.z[i] = b.take<float>(n);
        w.a[i] = b.take<float>(n);
        w.mean[i] = b.take<float>(L.fout);
        w.invstd[i] = b.take<float>(L.fout);
        w.scale[i] = b.take<float>(L.fout);
        w.shift[i] = b.take<float>(L.fout);
      } else {
        w.z[i] = w.a[i] = nullptr;  // last layer writes y directly
        w.mean[i] = w.invstd[i] = w.scale[i] = w.shift[i] = nullptr;
      }
    }
    w.fc_out = b.take<float>((size_t)B * m->fc_out);
  }
  w.bytes = b.off;
  return w;
}

struct BwdMap {
  float* G[4];
  float* U;
  float* dwp;
  double* sums;
  unsigned char* wpack;   // packed fp16 K-blocks of the backward-data conv (or of one W_k^T for the dT GEMM fallback)
  size_t wpack_bytes;
  unsigned char* wpack_iso;  // combined transposed weights of the isolated rows (padding-vertex elision)
  float* thin;               // scratch of the thin head's backward
  float* a_scale;         // power-of-two gradient scale (device scalar)
  size_t bytes;
};
BwdMap map_scratch(const p2m_model* m, int B, void* base) {
  BwdMap w;
  Sizes s = model_sizes(m, B);
  Bump b(base);
  for (int i = 0; i < 4; ++i) w.G[i] = b.take<float>(s.max_act);
  w.U = b.take<float>(s.max_U);
  w.dwp = b.take<float>(std::max(s.max_w, (size_t)1));
  w.sums = b.take<double>(2 * (size_t)s.max_f + 2 * (size_t)m->fc_out);
  w.wpack_bytes = umma_wpack_bytes(256, 256);   // backward-data conv image (>= the plain image of one W_k^T)
  w.wpack = b.take<unsigned char>(w.wpack_bytes);
  w.wpack_iso = b.take<unsigned char>(umma_plain_pack_bytes(256, 256));
  w.thin = b.take<float>(s.max_thin);
  w.a_scale = b.take<float>(4);
  w.bytes = b.off;
  return w;
}

// ---- one conv layer, linear part + epilogue -------------------------------------------------
// y = epilogue( [T0|T1|T2](x) * Wp^T )
bool conv_on_tensor_cores(const p2m_model* m, const Layer& L, const unsigned char* wpack) {
  return m->precision == P2M_PREC_FP16X3_TC && wpack != nullptr && umma_conv_supported(m->levels[L.level], L.fin, L.fout);
}
int conv_linear(p2m_model* m, const Layer& L, int B, const float* x, int in_unpool, const float* w_ref, float* T,
                float* wp, unsigned char* wpack, const Epilogue& ep, float* y, cudaStream_t s,
                const float* head_wt = nullptr, float* head_z = nullptr, bool keep_wp = true, bool may_elide = false,
                int iso_mode = 0 /* 0: every isolated row, 1: class representatives only, 2: none */) {
  const int rows = B * L.V;
  const DevLevel& g = m->levels[L.level];
  // k-major copy of the weights: what the SIMT GEMM reads, and (training, keep_wp) what backward's SIMT dT GEMM reads
  if (keep_wp || !conv_on_tensor_cores(m, L, wpack)) P2M_TRY(launch_permute_w(w_ref, wp, L.fout, L.fin, s));
  if (conv_on_tensor_cores(m, L, wpack)) {
    P2M_TRY(launch_umma_pack_weights(w_ref, L.fin, L.fout, wpack, s));
    UmmaConvArgs a;
    a.trace = m->trace;
    if (a.trace != nullptr) {  // trace builds only: P2M_TRACE_V / P2M_TRACE_UNPOOL pick the layer whose launch is logged
      const char* tv = getenv("P2M_TRACE_V");
      const char* tu = getenv("P2M_TRACE_UNPOOL");
      const char* tf = getenv("P2M_TRACE_FOUT");
      if ((tv && atoi(tv) != L.V) || (tu && atoi(tu) != in_unpool) || (tf && atoi(tf) != L.fout)) a.trace = nullptr;
    }
    a.head_wt = head_wt;
    a.head_z = head_z;
    // Padding-vertex elision (DevLevel::n_iso): connected rows through the conv on index-list tiles, isolated rows
    // through a plain GEMM with the combined weights.  Needs the T buffer of the network schedules (3 Fin wide: the
    // packed combined weights live behind the T1 part).
    const bool elide = may_elide && m->elide_padding && m->split_t1 && T != nullptr && g.n_iso > 0 &&
                       rows >= 2 * L.fout && (m->elide_padding >= 2 || 5LL * g.n_iso >= 2LL * g.V);
    if (m->split_t1 && T != nullptr) {  // first sparse product as its own pass (T doubles as the T1 buffer)
      P2M_TRY(launch_cheb_t1(g, x, in_unpool, B, L.fin, T, s, elide ? &g.real_tiles : nullptr));
      a.t1 = T;
    }
    a.g = &g;
    a.x = x;
    a.in_unpool = in_unpool;
    a.batch = B;
    a.fin = L.fin;
    a.fout = L.fout;
    a.wpack = wpack;
    a.ep = ep;
    a.y = y;
    if (!elide) return launch_umma_conv(a, m->kernel_status, m->zero_row, m->sm_count, s);
    a.tiles = &g.real_tiles;
    P2M_TRY(launch_umma_conv(a, m->kernel_status, m->zero_row, m->sm_count, s));
    if (iso_mode == 2) return P2M_OK;  // nothing the caller reads depends on the isolated rows (gathered eval output)
    const bool reps_only = (iso_mode == 1 && g.n_rep > 0);
    unsigned char* w_iso = reinterpret_cast<unsigned char*>(T + (size_t)rows * L.fin);
    P2M_TRY(launch_umma_pack_iso(w_ref, g.iso_diag, L.fin, L.fout, w_iso, s));
    a.t1 = nullptr;
    a.plain = 1;
    a.tiles = reps_only ? &g.rep_tiles : &g.iso_tiles;
    a.wpack = w_iso;
    return launch_umma_conv(a, m->kernel_status, m->zero_row, m->sm_count, s);
  }
  if (head_z != nullptr) {
    set_error("conv_linear: fused head requested off the tensor-core path");
    return P2M_ERR_INVALID;
  }
  if (thin_conv_supported(L.fin, L.fout) && ep.res == nullptr &&
      thin_conv_scratch_floats(rows, L.fin) <= (size_t)rows * 3 * L.fin) {
    return launch_thin_conv(g, x, in_unpool, rows, L.fin, L.fout, w_ref, ep, T, y, s);  // T doubles as scratch
  }
  P2M_TRY(launch_cheb_basis(g, x, in_unpool, rows, L.fin, T, s));
  P2M_TRY(launch_gemm(T, 3 * L.fin, wp, 3 * L.fin, 0, y, L.fout, rows, L.fout, 3 * L.fin, ep, s));
  return P2M_OK;
}

// The default elision policy (elide_padding == 1): levels that have the tile families and where at least 40 % of
// the rows are isolated.
inline bool policy_elided(const DevLevel& g) { return g.n_iso > 0 && 5LL * g.n_iso >= 2LL * g.V; }

// Classes of identical isolated rows (eval mode, DevLevel::rep_tiles).  Levels are ordered fine -> coarse, the joint
// graph last; the parent of row r of mesh level k is row r >> 1 of level k + 1 (nearest x2 unpool, meshnet.py:71-78).
// An isolated row is a REPRESENTATIVE if its parent is a connected row (nothing to share), or if it is the left
// child of a parent whose value is computed (any row of a level that is not elided, a representative otherwise);
// every other isolated row equals a representative: its left sibling, or the left child of its parent's
// representative.  Requires what the reference's binary-tree reorder guarantees (lib/coarsening.py:214-258: fake
// nodes are added bottom-up, so both children of a fake node are fake); if a level violates it the classes are
// simply not built (n_rep stays 0) and every isolated row is computed.
int build_padding_classes(p2m_model* m, const p2m_model_desc_t* d) {
  const int n_mesh = d->n_levels - 1;  // the last level is the joint graph
  std::vector<std::vector<char>> iso(n_mesh);
  for (int k = 0; k < n_mesh; ++k) {
    const int V = d->level_size[k];
    const int32_t* rp = d->rowptr[k];
    iso[k].assign(V, 0);
    for (int v = 0; v < V; ++v) iso[k][v] = (rp[v + 1] - rp[v] == 1 && d->colidx[k][rp[v]] == v) ? 1 : 0;
  }
  std::vector<std::vector<int>> rep_of(n_mesh);  // per elided level: representative of each isolated row (itself if rep)
  for (int k = n_mesh - 1; k >= 0; --k) {
    DevLevel& g = m->levels[k];
    if (!policy_elided(g)) continue;
    const int V = g.V;
    const bool has_parent = (k + 1 < n_mesh) && (d->level_size[k + 1] * 2 == V);
    const bool parent_elided = has_parent && policy_elided(m->levels[k + 1]);
    std::vector<int>& ro = rep_of[k];
    ro.assign(V, -1);
    std::vector<int> reps, cdst, csrc;
    bool ok = true;
    for (int r = 0; r < V && ok; ++r) {
      if (!iso[k][r]) continue;
      const int p = r >> 1;
      if (!has_parent || !iso[k + 1][p]) {
        ro[r] = r;
      } else {
        if (!iso[k][r ^ 1]) ok = false;  // both children of a fake vertex must be fake
        const bool parent_computed = !parent_elided || rep_of[k + 1][p] == p;
        if (parent_computed) ro[r] = r & ~1;
        else ro[r] = 2 * rep_of[k + 1][p];
        if (ro[r] < 0 || ro[r] >= V || !iso[k][ro[r]]) ok = false;
      }
      if (ro[r] == r) reps.push_back(r);
      else {
        cdst.push_back(r);
        csrc.push_back(ro[r]);
      }
    }
    for (size_t i = 0; i < csrc.size() && ok; ++i)
      if (ro[csrc[i]] != csrc[i]) ok = false;  // a representative represents itself
    if (!ok || cdst.empty()) {
      ro.assign(V, -1);  // treat the level as fully computed
      for (int r = 0; r < V; ++r)
        if (iso[k][r]) ro[r] = r;
      continue;
    }
    P2M_TRY(build_index_tiles(reps, d->rowptr[k], d->colidx[k], d->values[k], V, &g.rep_tiles, &m->owned));
    P2M_TRY(upload(m, cdst, &g.copy_dst));
    P2M_TRY(upload(m, csrc, &g.copy_src));
    g.n_rep = (int)reps.size();
    g.n_copy = (int)cdst.size();
  }
  // a level's classes assume that its elided parent level is deduplicated too: keep them only in a chain from the
  // finest level down (n_rep == 0 on a level switches its children back to "parent fully computed" == still valid,
  // because a fully computed parent only adds valid rows)
  return P2M_OK;
}

int check_params(const p2m_model* m, const p2m_params_t* p, bool need_running) {
  if (!p || !p->fc_w || !p->fc_b || !p->cl_w || !p->cl_b || !p->bn_w || !p->bn_b) {
    set_error("params: null table");
    return P2M_ERR_INVALID;
  }
  for (size_t i = 0; i < m->layers.size(); ++i) {
    if (!p->cl_w[i] || !p->cl_b[i]) {
      set_error("params: null conv weight/bias for layer " + std::to_string(i));
      return P2M_ERR_INVALID;
    }
    if (m->layers[i].bn) {
      if (!p->bn_w[i] || !p->bn_b[i] || (need_running && (!p->bn_rm || !p->bn_rv || !p->bn_rm[i] || !p->bn_rv[i]))) {
        set_error("params: null BatchNorm tensor for layer " + std::to_string(i));
        return P2M_ERR_INVALID;
      }
    }
  }
  return P2M_OK;
}

}  // namespace

// =====================================================================================
extern "C" {

const char* p2m_last_error(void) { return g_error.c_str(); }
const char* p2m_version(void) { return "pose2mesh_release_b200 0.1 (sm_100a)"; }
int64_t p2m_launch_count(void) { return g_launches; }
void p2m_launch_count_reset(void) { g_launches = 0; }

int p2m_model_create(const p2m_model_desc_t* d, p2m_model_t** out) {
  if (!d || !out || d->n_levels < 1 || (d->n_blocks != 0 && (d->n_blocks < 3 || d->n_levels < 2))) {
    set_error("model_create: bad descriptor");
    return P2M_ERR_INVALID;
  }
  // n_blocks == 0: graph-only handle (levels without a channel plan) for the single-layer entry points
  if (d->n_blocks != 0 && d->n_levels != d->n_blocks - 1) {
    set_error("model_create: need n_levels == n_blocks - 1 (one level per block; the last block re-uses the finest)");
    return P2M_ERR_INVALID;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || d->device >= ndev) {
    set_error("model_create: no usable CUDA device (this library has no CPU path)");
    cudaGetLastError();
    return P2M_ERR_NOGPU;
  }
  cudaDeviceProp prop;
  P2M_CUDA_OK(cudaGetDeviceProperties(&prop, d->device));
  if (prop.major != 10) {
    set_error(std::string("model_create: device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
              ", this library is built for sm_100a only");
    return P2M_ERR_NOGPU;
  }
  DeviceGuard guard(d->device);
  p2m_model* m = new p2m_model();
  m->device = d->device;
  m->sm_count = prop.multiProcessorCount;
  // ---- levels: CSR with relative offsets
  for (int l = 0; l < d->n_levels; ++l) {
    DevLevel g;
    g.V = d->level_size[l];
    const int32_t* rp = d->rowptr[l];
    g.nnz = rp[g.V];
    std::vector<int> rowptr(rp, rp + g.V + 1), rel(g.nnz);
    std::vector<float> val(d->values[l], d->values[l] + g.nnz);
    for (int v = 0; v < g.V; ++v) {
      g.max_row_nnz = std::max(g.max_row_nnz, rp[v + 1] - rp[v]);
      for (int p = rp[v]; p < rp[v + 1]; ++p) {
        int c = d->colidx[l][p];
        if (c < 0 || c >= g.V) {
          set_error("model_create: column index out of range");
          p2m_model_destroy(m);
          return P2M_ERR_INVALID;
        }
        rel[p] = c - v;
      }
    }
    int st;
    if ((st = upload(m, rowptr, &g.rowptr)) || (st = upload(m, rel, &g.reloff)) || (st = upload(m, val, &g.val)) ||
        (st = build_umma_level_meta(rp, d->colidx[l], d->values[l], g.V, &g, &m->owned))) {
      p2m_model_destroy(m);
      return st;
    }
    m->levels.push_back(g);
  }
  if (d->n_blocks != 0) {
    int st = build_padding_classes(m, d);
    if (st) {
      p2m_model_destroy(m);
      return st;
    }
  }
  {
    std::vector<float> zrow(64, 0.f);
    int st = upload(m, zrow, &m->zero_row);
    void* hp = nullptr;
    if (!st && (cudaHostAlloc(&hp, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess ||
                cudaHostGetDevicePointer(reinterpret_cast<void**>(&m->kernel_status), hp, 0) != cudaSuccess)) {
      set_error("model_create: cannot allocate the mapped status word");
      if (hp) cudaFreeHost(hp);
      st = P2M_ERR_CUDA;
    }
    if (st) {
      p2m_model_destroy(m);
      return st;
    }
    m->status_host = static_cast<volatile int*>(hp);
    *m->status_host = 0;
  }
  // ---- plan (meshnet.py:21-33, 86-94)
  const int nb = d->n_blocks;
  int off = 0, li = 0;
  for (int b = 0; b < nb; ++b) {
    const int32_t* ch = d->block_chans + off;
    const int len = d->block_len[b];
    if (len < 2) {
      set_error("model_create: block with < 2 channel entries");
      p2m_model_destroy(m);
      return P2M_ERR_INVALID;
    }
    Block blk{};
    blk.first_layer = li;
    blk.n_layers = len - 1;
    blk.level = (b == nb - 1) ? 0 : d->n_levels - 1 - b;
    blk.has_residual = (b >= 1 && b <= nb - 2);
    blk.out_unpool = (b >= 1 && b < nb - 2);
    blk.in_unpool = (b >= 2 && b <= nb - 2);
    blk.cin = ch[0];
    blk.cout = ch[len - 1];
    for (int j = 0; j < len - 1; ++j) {
      Layer L{};
      L.level = blk.level;
      L.V = m->levels[L.level].V;
      L.fin = ch[j];
      L.fout = ch[j + 1];
      const bool last = (b == nb - 1) && (j == len - 2);
      L.bn = !last;
      L.relu = !last;
      L.block = b;
      L.pos = j;
      L.block_end = (j == len - 2);
      m->layers.push_back(L);
      ++li;
    }
    if (blk.has_residual) {
      int st = build_interp(m, blk.cin, blk.cout, &blk.interp);
      if (st) {
        p2m_model_destroy(m);
        return st;
      }
    }
    m->blocks.push_back(blk);
    off += len;
  }
  // consistency: unpool doubles the level size; block b+1 input channels == block b output channels
  for (int b = 1; b < nb; ++b) {
    const Block& p = m->blocks[b - 1];
    const Block& c = m->blocks[b];
    bool ok = (c.cin == p.cout);
    if (b >= 2) {
      int vp = m->levels[p.level].V, vc = m->levels[c.level].V;
      ok = ok && (p.out_unpool ? (vc == 2 * vp) : (vc == vp));
    }
    if (!ok) {
      set_error("model_create: inconsistent hierarchy / channel plan at block " + std::to_string(b));
      p2m_model_destroy(m);
      return P2M_ERR_INVALID;
    }
  }
  if (nb == 0) {
    *out = m;
    return P2M_OK;
  }
  m->n_joint = m->levels.back().V;
  m->cin = m->blocks[0].cin;
  m->cout = m->blocks[nb - 1].cout;
  m->fc_in = m->n_joint * m->blocks[0].cout;
  m->fc_out = m->levels[m->blocks[1].level].V * m->blocks[1].cin;
  *out = m;
  return P2M_OK;
}

void p2m_model_destroy(p2m_model_t* m) {
  if (!m) return;
  DeviceGuard guard(m->device);
  for (void* p : m->owned) cudaFree(p);
  if (m->status_host) cudaFreeHost(const_cast<int*>(m->status_host));
  for (cudaEvent_t e : m->ev_beg) cudaEventDestroy(e);
  for (cudaEvent_t e : m->ev_end) cudaEventDestroy(e);
  delete m;
}

int p2m_model_num_layers(const p2m_model_t* m) { return m ? (int)m->layers.size() : 0; }

int p2m_model_layer_info(const p2m_model_t* m, int layer, int32_t out[6]) {
  if (!m || layer < 0 || layer >= (int)m->layers.size()) {
    set_error("layer_info: bad layer");
    return P2M_ERR_INVALID;
  }
  const Layer& L = m->layers[layer];
  out[0] = L.level; out[1] = L.V; out[2] = L.fin; out[3] = L.fout; out[4] = L.bn; out[5] = L.relu;
  return P2M_OK;
}

int p2m_debug_kernel_status(p2m_model_t* m, int32_t* out) {
  if (!m || !out) {
    set_error("debug_kernel_status: bad argument");
    return P2M_ERR_INVALID;
  }
  DeviceGuard guard(m->device);
  P2M_CUDA_OK(cudaDeviceSynchronize());
  *out = m->status_host ? *m->status_host : 0;
  return P2M_OK;
}

// Debug: route the tcgen05 conv kernel's CTA-0 event log into `dev_buf` (device, 8*512 int64) or disable (NULL).
// Only in libraries built with -DP2M_UMMA_TRACE (P2M_TRACE=1 python -m pose2mesh_release_b200.build --force).
int p2m_debug_set_trace(p2m_model_t* m, void* dev_buf) {
  if (!m) return P2M_ERR_INVALID;
#ifdef P2M_UMMA_TRACE
  m->trace = static_cast<long long*>(dev_buf);
  return P2M_OK;
#else
  if (dev_buf == nullptr) return P2M_OK;
  set_error("debug_set_trace: this library was built without P2M_UMMA_TRACE");
  return P2M_ERR_INVALID;
#endif
}

// Debug / ablation: 1 (default) = two-pass tcgen05 conv (k_cheb_t1 + conv with given T1), 0 = fully fused conv.
int p2m_debug_set_split_t1(p2m_model_t* m, int enable) {
  if (!m) return P2M_ERR_INVALID;
  m->split_t1 = enable ? 1 : 0;
  return P2M_OK;
}
int p2m_debug_set_elide_padding(p2m_model_t* m, int enable) {
  if (!m) return P2M_ERR_INVALID;
  m->elide_padding = enable < 0 ? 0 : (enable > 2 ? 2 : enable);
  return P2M_OK;
}
int p2m_debug_set_dedup_padding(p2m_model_t* m, int enable) {
  if (!m) return P2M_ERR_INVALID;
  m->dedup_padding = enable ? 1 : 0;
  return P2M_OK;
}
int p2m_debug_set_dw_swap(p2m_model_t* m, int enable) {
  if (!m) return P2M_ERR_INVALID;
  m->dw_swap = enable ? 1 : 0;
  return P2M_OK;
}
int p2m_debug_set_fuse_head(p2m_model_t* m, int enable) {
  if (!m) return P2M_ERR_INVALID;
  m->fuse_head = enable ? 1 : 0;
  return P2M_OK;
}

int p2m_model_set_profiling(p2m_model_t* m, int enable) {
  if (!m) {
    set_error("set_profiling: bad argument");
    return P2M_ERR_INVALID;
  }
  DeviceGuard guard(m->device);
  if (enable && m->ev_beg.empty()) {
    m->ev_beg.resize(m->layers.size());
    m->ev_end.resize(m->layers.size());
    for (size_t i = 0; i < m->layers.size(); ++i) {
      P2M_CUDA_OK(cudaEventCreate(&m->ev_beg[i]));
      P2M_CUDA_OK(cudaEventCreate(&m->ev_end[i]));
    }
  }
  m->profiling = enable ? 1 : 0;
  return P2M_OK;
}

int p2m_model_layer_times_ms(p2m_model_t* m, float* out, int n) {
  if (!m || !out || n < (int)m->layers.size() || m->ev_beg.empty()) {
    set_error("layer_times_ms: profiling was not enabled or buffer too small");
    return P2M_ERR_INVALID;
  }
  DeviceGuard guard(m->device);
  for (size_t i = 0; i < m->layers.size(); ++i) {
    P2M_CUDA_OK(cudaEventSynchronize(m->ev_end[i]));
    P2M_CUDA_OK(cudaEventElapsedTime(&out[i], m->ev_beg[i], m->ev_end[i]));
  }
  return P2M_OK;
}

int p2m_model_set_precision(p2m_model_t* m, int precision) {
  if (!m || (precision != P2M_PREC_FP32_SIMT && precision != P2M_PREC_FP16X3_TC)) {
    set_error("set_precision: bad argument");
    return P2M_ERR_INVALID;
  }
  m->precision = precision;
  return P2M_OK;
}

size_t p2m_meshnet_workspace_bytes(const p2m_model_t* m, int batch, int training) {
  if (!m || batch <= 0 || m->layers.empty()) return 0;
  return map_workspace(m, batch, training, nullptr).bytes;
}
size_t p2m_meshnet_backward_scratch_bytes(const p2m_model_t* m, int batch) {
  if (!m || batch <= 0 || m->layers.empty()) return 0;
  return map_scratch(m, batch, nullptr).bytes;
}
size_t p2m_meshnet_host_io_bytes(const p2m_model_t* m, int batch) {
  if (!m || batch <= 0 || m->layers.empty()) return 0;
  return align_up((size_t)batch * m->n_joint * m->cin * 4) + align_up((size_t)batch * m->levels[0].V * m->cout * 4);
}

// -------------------------------------------------------------------------------------
static int meshnet_forward_impl(p2m_model_t* m, const p2m_params_t* P, const float* x, float* y, int B, int training,
                                void* workspace, size_t workspace_bytes, p2m_stream_t stream, int gathered) {
  if (!m || !x || !y || B <= 0 || !workspace || m->layers.empty()) {
    set_error("meshnet_forward: bad argument");
    return P2M_ERR_INVALID;
  }
  P2M_TRY(check_params(m, P, true));
  P2M_TRY(check_kernel_status(m, "meshnet_forward"));
  DeviceGuard guard(m->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  WsMap w = map_workspace(m, B, training, workspace);
  if (w.bytes > workspace_bytes) {
    set_error("meshnet_forward: workspace too small (" + std::to_string(workspace_bytes) + " < " +
              std::to_string(w.bytes) + ")");
    return P2M_ERR_WORKSPACE;
  }
  const int nb = (int)m->blocks.size();
  const int nl = (int)m->layers.size();
  // isolated (padding) rows in eval mode: only class representatives (DevLevel::rep_tiles), or — when the caller
  // takes the gathered real vertices — none at all: no connected row ever reads an isolated one
  const int iso_mode = (training || !m->dedup_padding || m->elide_padding < 1) ? 0 : (gathered ? 2 : 1);
  const float* cur = x;
  int cur_unpool = 0;
  int cur_buf = -1;  // rotating buffer id holding `cur` (eval)
  float* head_z = nullptr;  // eval: Z of the thin head, produced by the previous layer's epilogue (see below)
  for (int b = 0; b < nb; ++b) {
    const Block& blk = m->blocks[b];
    const float* block_in = cur;
    const int block_in_unpool = cur_unpool;
    const int block_in_buf = cur_buf;
    for (int j = 0; j < blk.n_layers; ++j) {
      const int li = blk.first_layer + j;
      const Layer& L = m->layers[li];
      const int rows = B * L.V;
      const bool last = (li == nl - 1);
      const bool with_res = L.block_end && blk.has_residual;
      if (!training) {
        Epilogue ep;
        float* scale = w.scale_scratch;
        float* shift = w.scale_scratch + L.fout;
        if (L.bn) {
          P2M_TRY(launch_bn_fold_eval(P->bn_w[li], P->bn_b[li], P->bn_rm[li], P->bn_rv[li], P->cl_b[li], scale, shift,
                                      L.fout, s));
          ep.scale = scale;
          ep.shift = shift;
        } else {
          ep.bias = P->cl_b[li];
        }
        ep.relu = L.relu;
        if (with_res) {
          ep.res = block_in;
          ep.res_F = blk.cin;
          ep.res_unpool = block_in_unpool;
          ep.res_i0 = blk.interp.i0;
          ep.res_i1 = blk.interp.i1;
          ep.res_lam = blk.interp.lam;
        }
        float* out;
        int out_buf = -1;
        if (last) {
          out = y;
          if (gathered) {
            if (!thin_conv_supported(L.fin, L.fout) || with_res) {
              set_error("meshnet_forward_vertices: the head layer is not on the fused-gather path");
              return P2M_ERR_INVALID;
            }
            ep.out_map = m->out_map;
            ep.out_rows = m->out_rows;
            ep.level_V = L.V;
          }
        } else {
          for (int c = 0; c < 3; ++c)
            if (c != cur_buf && c != block_in_buf) {
              out_buf = c;
              break;
            }
          out = w.rot[out_buf];
        }
        if (m->profiling) P2M_CUDA_OK(cudaEventRecord(m->ev_beg[li], s));
        // Fused head: when the next layer is the network's thin head (64 -> 3, same block, no residual) and this
        // layer runs on the tensor cores, its epilogue writes Z = act(y) W' (12 floats per row) instead of y, and
        // the head shrinks to its two 4-wide sparse products: the 64-wide activation never reaches HBM.
        bool fuse_head = false;
        if (m->fuse_head && !last && li + 1 == nl - 1 && j + 1 < blk.n_layers && !with_res && !blk.has_residual &&
            L.fout == 64 && rows >= 64 && conv_on_tensor_cores(m, L, w.wpack)) {
          const Layer& H = m->layers[li + 1];
          fuse_head = thin_conv_supported(H.fin, H.fout) && H.fin == L.fout && H.V == L.V;
        }
        if (head_z != nullptr) {  // this IS the head, its Z is already there
          P2M_TRY(launch_thin_tail(m->levels[L.level], rows, L.fout, head_z, head_z + (size_t)rows * 12, ep, out, s));
          head_z = nullptr;
        } else if (fuse_head) {
          float* Z = out;  // [rows][12] | U [rows][4] | W' [64][12] inside this layer's (unused) output buffer
          float* wt = Z + (size_t)rows * 16;
          P2M_TRY(launch_thin_prep(P->cl_w[li + 1], L.fout, m->layers[li + 1].fout, wt, s));
          P2M_TRY(conv_linear(m, L, B, cur, cur_unpool, P->cl_w[li], w.T, w.wp_scratch, w.wpack, ep, out, s, wt, Z,
                              false, true, iso_mode));
          head_z = Z;
        } else {
          P2M_TRY(conv_linear(m, L, B, cur, cur_unpool, P->cl_w[li], w.T, w.wp_scratch, w.wpack, ep, out, s, nullptr,
                              nullptr, false, true, iso_mode));
        }
        if (m->profiling) P2M_CUDA_OK(cudaEventRecord(m->ev_end[li], s));
        cur = out;
        cur_buf = out_buf;
        cur_unpool = 0;
      } else {
        Epilogue ep;
        ep.bias = P->cl_b[li];
        float* z = last ? y : w.z[li];
        P2M_TRY(conv_linear(m, L, B, cur, cur_unpool, P->cl_w[li], w.T, w.wp[li], w.wpack, ep, z, s, nullptr, nullptr,
                            true, true));
        if (L.bn) {
          P2M_TRY(launch_col_stats(z, rows, L.fout, w.sums, s));
          P2M_TRY(launch_bn_finalize(w.sums, rows, L.fout, P->bn_w[li], P->bn_b[li], P->bn_rm[li], P->bn_rv[li],
                                     P->bn_nbt ? P->bn_nbt[li] : nullptr, w.mean[li], w.invstd[li], w.scale[li],
                                     w.shift[li], s));
          P2M_TRY(launch_affine_act(z, rows, L.fout, w.scale[li], w.shift[li], L.relu, with_res ? block_in : nullptr,
                                    blk.cin, block_in_unpool, with_res ? &blk.interp : nullptr, w.a[li], s));
          cur = w.a[li];
        } else {
          cur = z;
        }
        cur_unpool = 0;
      }
    }
    if (b == 0) {  // fc: joints -> coarsest mesh level (meshnet.py:104-106)
      Epilogue ep;
      ep.bias = P->fc_b;
      float* out;
      if (!training) {
        int out_buf = -1;
        for (int c = 0; c < 3; ++c)
          if (c != cur_buf) {
            out_buf = c;
            break;
          }
        out = w.rot[out_buf];
        cur_buf = out_buf;
      } else {
        out = w.fc_out;
      }
      if (m->precision == P2M_PREC_FP16X3_TC && w.fc_apack != nullptr)  // dense GEMM on tcgen05 (fp16x3)
        P2M_TRY(launch_umma_gemm(cur, P->fc_w, B, m->fc_out, m->fc_in, ep, out, w.fc_apack, w.fc_wpack, m->kernel_status,
                                 m->sm_count, s));
      else
        P2M_TRY(launch_gemm(cur, m->fc_in, P->fc_w, m->fc_in, 0, out, m->fc_out, B, m->fc_out, m->fc_in, ep, s));
      cur = out;
      cur_unpool = 0;
    } else if (blk.out_unpool) {
      cur_unpool = 1;  // nearest x2 unpool is virtual: the next block reads row r>>1
    }
  }
  if (iso_mode == 1 && m->levels[0].n_copy > 0) {
    // fill the output rows of the isolated vertices that were represented by another row of their class
    const DevLevel& g0 = m->levels[0];
    P2M_TRY(launch_copy_rows(y, B, g0.V, m->cout, g0.copy_dst, g0.copy_src, g0.n_copy, s));
  }
  return P2M_OK;
}

int p2m_meshnet_forward(p2m_model_t* m, const p2m_params_t* P, const float* x, float* y, int B, int training,
                        void* workspace, size_t workspace_bytes, p2m_stream_t stream) {
  return meshnet_forward_impl(m, P, x, y, B, training, workspace, workspace_bytes, stream, 0);
}

int p2m_model_set_output_gather(p2m_model_t* m, const int32_t* vertex_of_slot, int n_slots) {
  if (!m || m->layers.empty() || !vertex_of_slot || n_slots <= 0 || n_slots > m->levels[0].V) {
    set_error("set_output_gather: bad argument");
    return P2M_ERR_INVALID;
  }
  const int V0 = m->levels[0].V;
  std::vector<int> map(V0, -1);
  for (int j = 0; j < n_slots; ++j) {
    const int v = vertex_of_slot[j];
    if (v < 0 || v >= V0 || map[v] >= 0) {
      set_error("set_output_gather: index out of range or repeated");
      return P2M_ERR_INVALID;
    }
    map[v] = j;
  }
  DeviceGuard guard(m->device);
  if (m->out_map == nullptr) {  // one [V0] map per handle, overwritten in place by later calls
    P2M_TRY(upload(m, map, &m->out_map));
  } else {
    // earlier forwards may still be reading the old map on their streams
    P2M_CUDA_OK(cudaDeviceSynchronize());
    P2M_CUDA_OK(cudaMemcpy(m->out_map, map.data(), sizeof(int) * V0, cudaMemcpyHostToDevice));
  }
  m->out_rows = n_slots;
  return P2M_OK;
}

int p2m_meshnet_forward_vertices(p2m_model_t* m, const p2m_params_t* P, const float* x, float* y_vertices, int B,
                                 void* workspace, size_t workspace_bytes, p2m_stream_t stream) {
  if (!m || !m->out_map) {
    set_error("meshnet_forward_vertices: call p2m_model_set_output_gather first");
    return P2M_ERR_INVALID;
  }
  return meshnet_forward_impl(m, P, x, y_vertices, B, 0, workspace, workspace_bytes, stream, 1);
}

static int forward_host_impl(p2m_model_t* m, const p2m_params_t* P, const float* x_host, float* y_host, int B,
                             void* workspace, size_t workspace_bytes, p2m_stream_t stream, int gathered) {
  if (!m || !x_host || !y_host || B <= 0 || !workspace || m->layers.empty() || (gathered && !m->out_map)) {
    set_error(gathered && m && !m->out_map ? "meshnet_forward_vertices_host: call p2m_model_set_output_gather first"
                                           : "meshnet_forward_host: bad argument");
    return P2M_ERR_INVALID;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t out_rows = gathered ? (size_t)m->out_rows : (size_t)m->levels[0].V;
  const size_t xb = (size_t)B * m->n_joint * m->cin * 4, yb = (size_t)B * out_rows * m->cout * 4;
  const size_t io = p2m_meshnet_host_io_bytes(m, B);
  const size_t need = p2m_meshnet_workspace_bytes(m, B, 0);
  if (workspace_bytes < need + io) {
    set_error("meshnet_forward_host: workspace too small");
    return P2M_ERR_WORKSPACE;
  }
  DeviceGuard guard(m->device);
  char* base = static_cast<char*>(workspace);
  float* xd = reinterpret_cast<float*>(base + need);
  float* yd = reinterpret_cast<float*>(base + need + align_up(xb));
  P2M_CUDA_OK(cudaMemcpyAsync(xd, x_host, xb, cudaMemcpyHostToDevice, s));
  P2M_TRY(meshnet_forward_impl(m, P, xd, yd, B, 0, workspace, need, stream, gathered));
  P2M_CUDA_OK(cudaMemcpyAsync(y_host, yd, yb, cudaMemcpyDeviceToHost, s));
  P2M_CUDA_OK(cudaStreamSynchronize(s));
  return check_kernel_status(m, "meshnet_forward_host");
}

int p2m_meshnet_forward_host(p2m_model_t* m, const p2m_params_t* P, const float* x_host, float* y_host, int B,
                             void* workspace, size_t workspace_bytes, p2m_stream_t stream) {
  return forward_host_impl(m, P, x_host, y_host, B, workspace, workspace_bytes, stream, 0);
}

int p2m_meshnet_forward_vertices_host(p2m_model_t* m, const p2m_params_t* P, const float* x_host, float* y_vertices_host,
                                      int B, void* workspace, size_t workspace_bytes, p2m_stream_t stream) {
  return forward_host_impl(m, P, x_host, y_vertices_host, B, workspace, workspace_bytes, stream, 1);
}

// -------------------------------------------------------------------------------------
int p2m_meshnet_backward(p2m_model_t* m, const p2m_params_t* P, const p2m_params_t* G, const float* x, const float* dy,
                         float* dx, int B, void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                         p2m_stream_t stream) {
  if (!m || !x || !dy || B <= 0 || !workspace || !scratch || m->layers.empty()) {
    set_error("meshnet_backward: bad argument");
    return P2M_ERR_INVALID;
  }
  P2M_TRY(check_params(m, P, false));
  P2M_TRY(check_params(m, G, false));
  P2M_TRY(check_kernel_status(m, "meshnet_backward"));
  DeviceGuard guard(m->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  WsMap w = map_workspace(m, B, 1, workspace);
  BwdMap sc = map_scratch(m, B, scratch);
  if (w.bytes > workspace_bytes || sc.bytes > scratch_bytes) {
    set_error("meshnet_backward: workspace/scratch too small");
    return P2M_ERR_WORKSPACE;
  }
  const int nb = (int)m->blocks.size();
  const float* g_cur = dy;
  int g_cur_buf = -2;  // -2: external (dy)
  int keep_buf = -1;   // buffer holding g_out of the block being processed (residual path)
  const float* keep_ptr = nullptr;
  auto free_buf = [&](int a, int b2, int c) {
    for (int i = 0; i < 4; ++i)
      if (i != a && i != b2 && i != c) return i;
    return -1;
  };
  for (int b = nb - 1; b >= 0; --b) {
    const Block& blk = m->blocks[b];
    // input of this block (physical tensor + unpool flag)
    const float* block_in;
    if (b == 0)
      block_in = x;
    else if (b == 1)
      block_in = w.fc_out;
    else
      block_in = w.a[m->blocks[b - 1].first_layer + m->blocks[b - 1].n_layers - 1];
    for (int j = blk.n_layers - 1; j >= 0; --j) {
      const int li = blk.first_layer + j;
      const Layer& L = m->layers[li];
      const DevLevel& g = m->levels[L.level];
      const int rows = B * L.V;
      const float* inp = (j == 0) ? block_in : w.a[li - 1];
      const int in_unpool = (j == 0) ? blk.in_unpool : 0;
      const float* g_z = g_cur;
      int gz_buf = g_cur_buf;
      if (L.block_end && blk.has_residual) {
        keep_buf = g_cur_buf;
        keep_ptr = g_cur;
      }
      const bool tc = (m->precision == P2M_PREC_FP16X3_TC);
      const bool need_dx = !(li == 0 && dx == nullptr);
      const bool res_here = (j == 0) && blk.has_residual;
      // which path takes this layer's weight / data gradients
      const bool thin = thin_conv_bwd_supported(L.fin, L.fout) && !in_unpool && !res_here && li > 0;
      const bool tc_dw = tc && !thin && umma_dw_supported(g, L.fin, L.fout);
      const bool tc_dx = tc && !thin && need_dx && m->split_t1 && umma_conv_supported(g, L.fout, L.fin) &&
                         umma_wpack_bytes(L.fout, L.fin) <= sc.wpack_bytes && (size_t)L.fout <= 3 * (size_t)L.fin;
      const bool tc_dt = tc && !thin && need_dx && !tc_dx && umma_conv_supported(g, L.fout, L.fin) &&
                         umma_plain_pack_bytes(L.fin, L.fout) <= sc.wpack_bytes;
      const bool dw_swapped = tc_dx && m->dw_swap && umma_dw_swapped_supported(g, L.fin, L.fout);
      const bool want_scale = tc_dw || tc_dx || tc_dt;
      bool have_scale = false;
      if (L.bn) {
        int tgt = (g_cur_buf >= 0 && g_cur_buf != keep_buf) ? g_cur_buf : free_buf(g_cur_buf, keep_buf, -1);
        P2M_TRY(launch_bn_relu_bwd(w.z[li], g_cur, rows, L.fout, P->bn_w[li], w.scale[li], w.shift[li], w.mean[li],
                                   w.invstd[li], L.relu, sc.sums, G->bn_w[li], G->bn_b[li], sc.G[tgt], s,
                                   want_scale ? sc.a_scale : nullptr));
        have_scale = want_scale;
        g_z = sc.G[tgt];
        gz_buf = tgt;
        // the bias of a conv in front of a BatchNorm has a mathematically zero gradient (the batch mean removes
        // it): db = sum_rows dz = 0 exactly, where the reference accumulates fp32 rounding noise
        P2M_TRY(launch_fill_zero(G->cl_b[li], sizeof(float) * L.fout, s));
      } else {
        P2M_TRY(launch_col_sum(g_z, rows, L.fout, sc.sums, G->cl_b[li], s));
      }
      if (want_scale && !have_scale) P2M_TRY(launch_absmax_scale(g_z, (long long)rows * L.fout, sc.a_scale, s));
      float* out = nullptr;
      int out_buf = -1;
      if (need_dx) {
        if (li == 0) {
          out = dx;
        } else {
          out_buf = free_buf(gz_buf, keep_buf, -1);
          out = sc.G[out_buf];
        }
      }
      if (thin) {
        // weights-first backward of the thin head: dW and dX from the 3-wide basis of dz, X read once
        P2M_TRY(launch_thin_conv_bwd(g, inp, rows, L.fin, L.fout, P->cl_w[li], g_z, sc.thin, out, G->cl_w[li],
                                     m->sm_count, s));
      } else {
        // dW.  tcgen05 path: the basis is rebuilt on chip by the forward's producers and contracted with the
        // (power-of-two scaled) dz tile by MN-major UMMAs; otherwise SIMT: materialise T, dWp = g_z^T T.
        if (dw_swapped) {
          // sum_rows dz (x) T_k(X) = sum_rows T_k(dz) (x) X  (L~ symmetric): the basis of the GRADIENT, whose first
          // sparse product the backward-data pass below needs anyway, contracted with plain tiles of the layer input
          P2M_TRY(launch_cheb_t1(g, g_z, 0, B, L.fout, w.T, s, nullptr));
          P2M_TRY(launch_fill_zero(G->cl_w[li], sizeof(float) * L.fout * 3 * L.fin, s));
          P2M_TRY(launch_umma_dw_swapped(g, inp, in_unpool, B, L.fin, L.fout, g_z, w.T, sc.a_scale, G->cl_w[li],
                                         m->kernel_status, m->sm_count, s));
        } else if (tc_dw) {
          P2M_TRY(launch_fill_zero(G->cl_w[li], sizeof(float) * L.fout * 3 * L.fin, s));
          P2M_TRY(launch_umma_dw(g, inp, in_unpool, B, L.fin, L.fout, g_z, sc.a_scale, G->cl_w[li], m->kernel_status,
                                 m->sm_count, s));
        } else {
          P2M_TRY(launch_cheb_basis(g, inp, in_unpool, rows, L.fin, w.T, s));
          P2M_TRY(launch_fill_zero(sc.dwp, sizeof(float) * L.fout * 3 * L.fin, s));
          P2M_TRY(launch_gemm_tn_atomic(g_z, L.fout, w.T, 3 * L.fin, sc.dwp, 3 * L.fin, rows, L.fout, 3 * L.fin, s));
          P2M_TRY(launch_unpermute_w(sc.dwp, G->cl_w[li], L.fout, L.fin, s));
        }
      }
      // dX
      if (need_dx && tc_dx) {
        // Backward-data IS a forward conv: dXl = [dz | L~dz | (2L~^2 - I)dz] W'^T with W'[f][o*3+k] = W[o][f*3+k]
        // (L~ symmetric) — the T1 pass and the tcgen05 conv kernel of the forward, run on dz (scaled into fp16's
        // range by a power of two), with the padding-vertex elision of the forward.  An identity residual gradient
        // is added in the epilogue; the pair-sum of the virtual unpool and a resampled residual need a finishing pass.
        const bool identity_res = res_here && blk.cin == blk.cout;
        const bool finish = in_unpool || (res_here && !identity_res);
        float* dst = finish ? sc.U : out;
        const bool elide = m->elide_padding && g.n_iso > 0 && rows >= 2 * L.fin &&
                           (m->elide_padding >= 2 || 5LL * g.n_iso >= 2LL * g.V);
        if (!dw_swapped)  // (the swapped dW above already left L~dz of every row in w.T)
          P2M_TRY(launch_cheb_t1(g, g_z, 0, B, L.fout, w.T, s, elide ? &g.real_tiles : nullptr));
        P2M_TRY(launch_umma_pack_weights_t(P->cl_w[li], L.fin, L.fout, sc.wpack, s));
        UmmaConvArgs a;
        a.g = &g;
        a.x = g_z;
        a.in_unpool = 0;
        a.batch = B;
        a.fin = L.fout;
        a.fout = L.fin;
        a.wpack = sc.wpack;
        a.t1 = w.T;
        a.a_scale = sc.a_scale;
        a.y = dst;
        if (identity_res) {
          a.ep.res = keep_ptr;
          a.ep.res_F = blk.cout;
          a.ep.res_unpool = 0;
          a.ep.res_i0 = blk.interp.i0;
          a.ep.res_i1 = blk.interp.i1;
          a.ep.res_lam = blk.interp.lam;
        }
        if (elide) a.tiles = &g.real_tiles;
        P2M_TRY(launch_umma_conv(a, m->kernel_status, m->zero_row, m->sm_count, s));
        if (elide) {
          P2M_TRY(launch_umma_pack_iso_t(P->cl_w[li], g.iso_diag, L.fin, L.fout, sc.wpack_iso, s));
          a.t1 = nullptr;
          a.plain = 1;
          a.tiles = &g.iso_tiles;
          a.wpack = sc.wpack_iso;
          P2M_TRY(launch_umma_conv(a, m->kernel_status, m->zero_row, m->sm_count, s));
        }
        if (finish)
          P2M_TRY(launch_dx_finish(dst, rows, L.fin, (res_here && !identity_res) ? keep_ptr : nullptr, blk.cout,
                                   (res_here && !identity_res) ? &blk.interp : nullptr, in_unpool, out, s));
      } else if (need_dx && !thin) {
        Epilogue none;
        // dT = g_z * Wp  ([rows, Fout] x [Fout, 3 Fin]).  tcgen05 fallback: three plain GEMMs (one per Chebyshev
        // order, N = Fin, K = Fout) with the gradient scaled into fp16 range by a power of two.
        if (tc_dt) {
          for (int k = 0; k < 3; ++k) {
            // B_k[n = f][kk = o] = W[o, f*3 + k]   (reference layout, lib/models/backbones/cheby_graph_conv.py:32-37)
            P2M_TRY(launch_umma_pack_plain(P->cl_w[li] + k, 3, 3LL * L.fin, L.fin, L.fout, sc.wpack, s));
            UmmaConvArgs a;
            a.g = &g;
            a.x = g_z;
            a.in_unpool = 0;
            a.batch = B;
            a.fin = L.fout;
            a.fout = L.fin;
            a.wpack = sc.wpack;
            a.y = w.T;
            a.plain = 1;
            a.a_scale = sc.a_scale;
            a.ldy = 3LL * L.fin;
            a.y_col0 = k * L.fin;
            P2M_TRY(launch_umma_conv(a, m->kernel_status, m->zero_row, m->sm_count, s));
          }
        } else {
          P2M_TRY(launch_gemm(g_z, L.fout, w.wp[li], 3 * L.fin, 1, w.T, 3 * L.fin, rows, 3 * L.fin, L.fout, none, s));
        }
        P2M_TRY(launch_cheb_basis_bwd(g, w.T, rows, L.fin, sc.U, res_here ? keep_ptr : nullptr, blk.cout,
                                      res_here ? &blk.interp : nullptr, in_unpool, out, s));
      }
      if (need_dx) {
        g_cur = out;
        g_cur_buf = out_buf;
      }
      if (j == 0) {
        keep_buf = -1;
        keep_ptr = nullptr;
      }
    }
    if (b == 1) {  // fc backward (meshnet.py:104-106)
      const float* a0 = w.a[m->blocks[0].first_layer + m->blocks[0].n_layers - 1];  // [B, fc_in]
      P2M_TRY(launch_col_sum(g_cur, B, m->fc_out, sc.sums, G->fc_b, s));
      P2M_TRY(launch_fill_zero(G->fc_w, sizeof(float) * (size_t)m->fc_out * m->fc_in, s));
      P2M_TRY(launch_gemm_tn_atomic(g_cur, m->fc_out, a0, m->fc_in, G->fc_w, m->fc_in, B, m->fc_out, m->fc_in, s));
      int out_buf = free_buf(g_cur_buf, -1, -1);
      Epilogue none;
      P2M_TRY(launch_gemm(g_cur, m->fc_out, P->fc_w, m->fc_in, 1, sc.G[out_buf], m->fc_in, B, m->fc_in, m->fc_out, none, s));
      g_cur = sc.G[out_buf];
      g_cur_buf = out_buf;
    }
  }
  return P2M_OK;
}

// -------------------------------------------------------------------------------------
size_t p2m_cheb_conv_workspace_bytes(const p2m_model_t* m, int level, int batch, int fin, int fout) {
  if (!m || level < 0 || level >= (int)m->levels.size()) return 0;
  size_t rows = (size_t)batch * m->levels[level].V;
  return align_up(rows * 3 * fin * 4) + align_up((size_t)fout * 3 * fin * 4) * 2 + align_up(rows * fin * 4) +
         align_up(rows * fout * 4) + align_up(2 * (size_t)std::max(fin, fout) * 8) + align_up(2 * (size_t)fout * 4) +
         align_up(umma_wpack_bytes(((fin + 31) / 32) * 32, fout) + 16) + ALIGN;
}

int p2m_cheb_conv_fwd(p2m_model_t* m, const p2m_conv_fwd_args_t* a, void* workspace, size_t workspace_bytes,
                      p2m_stream_t stream) {
  if (!m || !a || !a->x || !a->weight || !a->bias || !a->y || a->level < 0 || a->level >= (int)m->levels.size()) {
    set_error("cheb_conv_fwd: bad argument");
    return P2M_ERR_INVALID;
  }
  if (workspace_bytes < p2m_cheb_conv_workspace_bytes(m, a->level, a->batch, a->fin, a->fout)) {
    set_error("cheb_conv_fwd: workspace too small");
    return P2M_ERR_WORKSPACE;
  }
  P2M_TRY(check_kernel_status(m, "cheb_conv_fwd"));
  DeviceGuard guard(m->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Layer L{};
  L.level = a->level;
  L.V = m->levels[a->level].V;
  L.fin = a->fin;
  L.fout = a->fout;
  const size_t rows = (size_t)a->batch * L.V;
  Bump b(workspace);
  float* T = b.take<float>(rows * 3 * L.fin);
  float* wp = b.take<float>((size_t)L.fout * 3 * L.fin);
  b.take<float>((size_t)L.fout * 3 * L.fin);
  b.take<float>(rows * L.fin);
  float* z = b.take<float>(rows * L.fout);
  double* sums = b.take<double>(2 * (size_t)std::max(L.fin, L.fout));
  float* sc = b.take<float>(2 * (size_t)L.fout);
  unsigned char* wpack = b.take<unsigned char>(umma_wpack_bytes(((L.fin + 31) / 32) * 32, L.fout) + 16);
  Epilogue ep;
  if (a->bn_mode == 0) {
    ep.bias = a->bias;
    ep.relu = a->relu;
    return conv_linear(m, L, a->batch, a->x, 0, a->weight, T, wp, wpack, ep, a->y, s);
  }
  if (!a->bn_weight || !a->bn_bias) {
    set_error("cheb_conv_fwd: BatchNorm parameters missing");
    return P2M_ERR_INVALID;
  }
  if (a->bn_mode == 1) {
    if (!a->bn_running_mean || !a->bn_running_var) {
      set_error("cheb_conv_fwd: running stats missing");
      return P2M_ERR_INVALID;
    }
    P2M_TRY(launch_bn_fold_eval(a->bn_weight, a->bn_bias, a->bn_running_mean, a->bn_running_var, a->bias, sc,
                                sc + L.fout, L.fout, s));
    ep.scale = sc;
    ep.shift = sc + L.fout;
    ep.relu = a->relu;
    return conv_linear(m, L, a->batch, a->x, 0, a->weight, T, wp, wpack, ep, a->y, s);
  }
  ep.bias = a->bias;
  P2M_TRY(conv_linear(m, L, a->batch, a->x, 0, a->weight, T, wp, wpack, ep, z, s));
  P2M_TRY(launch_col_stats(z, (int)rows, L.fout, sums, s));
  P2M_TRY(launch_bn_finalize(sums, (int)rows, L.fout, a->bn_weight, a->bn_bias, a->bn_running_mean, a->bn_running_var,
                             a->bn_num_batches_tracked, a->save_mean, a->save_invstd, sc, sc + L.fout, s));
  P2M_TRY(launch_affine_act(z, (int)rows, L.fout, sc, sc + L.fout, a->relu, nullptr, 0, 0, nullptr, a->y, s));
  return P2M_OK;
}

int p2m_cheb_conv_bwd(p2m_model_t* m, const p2m_conv_bwd_args_t* a, void* workspace, size_t workspace_bytes,
                      p2m_stream_t stream) {
  if (!m || !a || !a->x || !a->weight || !a->dz || !a->dweight || !a->dbias || a->level < 0 ||
      a->level >= (int)m->levels.size()) {
    set_error("cheb_conv_bwd: bad argument");
    return P2M_ERR_INVALID;
  }
  if (workspace_bytes < p2m_cheb_conv_workspace_bytes(m, a->level, a->batch, a->fin, a->fout)) {
    set_error("cheb_conv_bwd: workspace too small");
    return P2M_ERR_WORKSPACE;
  }
  P2M_TRY(check_kernel_status(m, "cheb_conv_bwd"));
  DeviceGuard guard(m->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const DevLevel& g = m->levels[a->level];
  const int fin = a->fin, fout = a->fout;
  const size_t rows = (size_t)a->batch * g.V;
  Bump b(workspace);
  float* T = b.take<float>(rows * 3 * fin);
  float* wp = b.take<float>((size_t)fout * 3 * fin);
  float* dwp = b.take<float>((size_t)fout * 3 * fin);
  float* U = b.take<float>(rows * fin);
  b.take<float>(rows * fout);
  double* sums = b.take<double>(2 * (size_t)std::max(fin, fout));
  float* sc2 = b.take<float>(2 * (size_t)fout);
  unsigned char* wpack = b.take<unsigned char>(umma_wpack_bytes(((fin + 31) / 32) * 32, fout) + 16);
  float* a_scale = sc2;  // device scalar for the tensor-core paths (the forward's scale/shift slot is free here)
  const bool tc = (m->precision == P2M_PREC_FP16X3_TC);
  bool have_scale = false;
  P2M_TRY(launch_col_sum(a->dz, (int)rows, fout, sums, a->dbias, s));
  if (tc && umma_dw_supported(g, fin, fout)) {
    P2M_TRY(launch_absmax_scale(a->dz, (long long)rows * fout, a_scale, s));
    have_scale = true;
    P2M_TRY(launch_fill_zero(a->dweight, sizeof(float) * fout * 3 * fin, s));
    P2M_TRY(launch_umma_dw(g, a->x, 0, a->batch, fin, fout, a->dz, a_scale, a->dweight, m->kernel_status, m->sm_count, s));
  } else {
    P2M_TRY(launch_cheb_basis(g, a->x, 0, (int)rows, fin, T, s));
    P2M_TRY(launch_fill_zero(dwp, sizeof(float) * fout * 3 * fin, s));
    P2M_TRY(launch_gemm_tn_atomic(a->dz, fout, T, 3 * fin, dwp, 3 * fin, (int)rows, fout, 3 * fin, s));
    P2M_TRY(launch_unpermute_w(dwp, a->dweight, fout, fin, s));
  }
  if (a->dx) {
    Epilogue none;
    if (tc && umma_conv_supported(g, fout, fin) && umma_plain_pack_bytes(fin, fout) <= umma_wpack_bytes(((fin + 31) / 32) * 32, fout)) {
      if (!have_scale) P2M_TRY(launch_absmax_scale(a->dz, (long long)rows * fout, a_scale, s));
      for (int k = 0; k < 3; ++k) {
        P2M_TRY(launch_umma_pack_plain(a->weight + k, 3, 3LL * fin, fin, fout, wpack, s));
        UmmaConvArgs u;
        u.g = &g;
        u.x = a->dz;
        u.in_unpool = 0;
        u.batch = a->batch;
        u.fin = fout;
        u.fout = fin;
        u.wpack = wpack;
        u.y = T;
        u.plain = 1;
        u.a_scale = a_scale;
        u.ldy = 3LL * fin;
        u.y_col0 = k * fin;
        P2M_TRY(launch_umma_conv(u, m->kernel_status, m->zero_row, m->sm_count, s));
      }
    } else {
      P2M_TRY(launch_permute_w(a->weight, wp, fout, fin, s));
      P2M_TRY(launch_gemm(a->dz, fout, wp, 3 * fin, 1, T, 3 * fin, (int)rows, 3 * fin, fout, none, s));
    }
    P2M_TRY(launch_cheb_basis_bwd(g, T, (int)rows, fin, U, nullptr, 0, nullptr, 0, a->dx, s));
  }
  return P2M_OK;
}

}  // extern "C"

// =====================================================================================
// Row f1 of SURVEY.md §8: what FlatPose2Mesh runs in front of MeshNet (lib/models/pose2mesh_net.py:16-22) —
// the PoseNet 2-D -> 3-D lifter (lib/models/posenet.py:41-87, eval mode: running-stat BatchNorm, dropout off) and
// the concat  pose_combine = cat(pose2d, pose3d / 1000)  that becomes MeshNet's input.
//   y  = x W1^T + b1                                                  [B, H]
//   per stage:  y += relu(bn2(relu(bn1(y)) Wa^T + ba)) Wb^T + bb
//   pose3d = y W2^T + b2                                              [B, 3J]
// fp32 FFMA GEMMs (k_gemm) with the BatchNorm / ReLU / residual fused into the epilogues; B rows only, so the
// 4 H x H weight matrices (64 MB each at H = 4096) dominate the traffic and are read once per call.
// =====================================================================================
namespace {
__global__ void __launch_bounds__(256) k_bn_relu_rows(const float* __restrict__ x, long long n, int F,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      const float* __restrict__ rm, const float* __restrict__ rv,
                                                      float* __restrict__ y) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int f = (int)(i % F);
  const float sc = gamma[f] / sqrtf(rv[f] + 1e-5f);
  y[i] = fmaxf(fmaf(x[i] - rm[f], sc, beta[f]), 0.f);
}
__global__ void __launch_bounds__(256) k_take_cols(const float* __restrict__ src, int ld, const float* __restrict__ bias,
                                                   int n_col, long long n, float* __restrict__ dst) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long r = i / n_col;
  const int c = (int)(i - r * n_col);
  dst[i] = src[r * ld + c] + bias[c];
}
__global__ void __launch_bounds__(256) k_pose_combine(const float* __restrict__ pose2d, const float* __restrict__ pose3d,
                                                      long long n_joint_rows, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (b, j)
  if (i >= n_joint_rows) return;
  out[i * 5 + 0] = pose2d[i * 2 + 0];
  out[i * 5 + 1] = pose2d[i * 2 + 1];
  out[i * 5 + 2] = pose3d[i * 3 + 0] / 1000.f;
  out[i * 5 + 3] = pose3d[i * 3 + 1] / 1000.f;
  out[i * 5 + 4] = pose3d[i * 3 + 2] / 1000.f;
}
}  // namespace

extern "C" {

size_t p2m_posenet_workspace_bytes(int batch, int hidden) {
  if (batch <= 0 || hidden <= 0) return 0;
  size_t n = 3 * align_up((size_t)batch * hidden * 4) + align_up(2 * (size_t)hidden * 4) + ALIGN;
  if (umma_gemm_supported(batch, hidden, hidden))  // operand images of the hidden x hidden GEMMs (tcgen05 path)
    n += align_up(umma_gemm_apack_bytes(batch, hidden)) + align_up(umma_gemm_wpack_bytes(hidden, hidden));
  return n;
}

int p2m_posenet_forward(const p2m_posenet_params_t* P, const float* pose2d, float* pose3d, float* pose_combine, int B,
                        void* workspace, size_t workspace_bytes, p2m_stream_t stream) {
  if (!P || !pose2d || !pose3d || B <= 0 || !workspace || P->num_joint <= 0 || P->hidden <= 0 || P->num_stage < 0 ||
      !P->w1_w || !P->w1_b || !P->w2_w || !P->w2_b) {
    set_error("posenet_forward: bad argument");
    return P2M_ERR_INVALID;
  }
  if (workspace_bytes < p2m_posenet_workspace_bytes(B, P->hidden)) {
    set_error("posenet_forward: workspace too small");
    return P2M_ERR_WORKSPACE;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int H = P->hidden, J = P->num_joint;
  Bump b(workspace);
  float* y = b.take<float>((size_t)B * H);
  float* a = b.take<float>((size_t)B * H);
  float* h = b.take<float>((size_t)B * H);
  float* sc = b.take<float>(2 * (size_t)H);
  int* status = b.take<int>(1);
  // The two H x H GEMMs of every stage run on tcgen05 (fp16x3, both operands streamed by cp.async.bulk:
  // launch_umma_gemm) when H allows; the thin first / last layers (K = 2J, N = 3J) stay on the fp32 SIMT GEMM.
  const bool tc = umma_gemm_supported(B, H, H);
  void* apack = tc ? b.take<unsigned char>(umma_gemm_apack_bytes(B, H)) : nullptr;
  void* wpack = tc ? b.take<unsigned char>(umma_gemm_wpack_bytes(H, H)) : nullptr;
  int sm_count = 148;
  if (tc) {
    int dev = 0;
    P2M_CUDA_OK(cudaGetDevice(&dev));
    P2M_CUDA_OK(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev));
    P2M_CUDA_OK(cudaMemsetAsync(status, 0, sizeof(int), s));
  }
  auto big_gemm = [&](const float* X, const float* Wm, const Epilogue& e, float* Y) -> int {
    if (tc) return launch_umma_gemm(X, Wm, B, H, H, e, Y, apack, wpack, status, sm_count, s);
    return launch_gemm(X, H, Wm, H, 0, Y, H, B, H, H, e, s);
  };
  Epilogue e1;
  e1.bias = P->w1_b;
  P2M_TRY(launch_gemm(pose2d, 2 * J, P->w1_w, 2 * J, 0, y, H, B, H, 2 * J, e1, s));
  for (int st = 0; st < P->num_stage; ++st) {
    const p2m_posenet_stage_t& S = P->stages[st];
    if (!S.w1_w || !S.w1_b || !S.w2_w || !S.w2_b || !S.bn1_w || !S.bn1_b || !S.bn1_rm || !S.bn1_rv || !S.bn2_w ||
        !S.bn2_b || !S.bn2_rm || !S.bn2_rv) {
      set_error("posenet_forward: null stage tensor");
      return P2M_ERR_INVALID;
    }
    // a = relu(bn1(y))
    const long long n = (long long)B * H;
    k_bn_relu_rows<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(y, n, H, S.bn1_w, S.bn1_b, S.bn1_rm, S.bn1_rv, a);
    P2M_LAUNCH_OK();
    // h = relu(bn2(a Wa^T + ba)): BatchNorm folded into the GEMM epilogue
    P2M_TRY(launch_bn_fold_eval(S.bn2_w, S.bn2_b, S.bn2_rm, S.bn2_rv, S.w1_b, sc, sc + H, H, s));
    Epilogue ea;
    ea.scale = sc;
    ea.shift = sc + H;
    ea.relu = 1;
    P2M_TRY(big_gemm(a, S.w1_w, ea, h));
    // y' = y + h Wb^T + bb  (written to `a`, then the buffers swap roles)
    Epilogue eb;
    eb.bias = S.w2_b;
    eb.res = y;
    eb.res_F = H;
    P2M_TRY(big_gemm(h, S.w2_w, eb, a));
    std::swap(y, a);
  }
  if (tc && 3 * J <= 64) {
    // the K = H reduction of the output layer on tcgen05 as well: N padded to 64 zero-weight columns (two CTAs of
    // the fp32 SIMT GEMM would walk the 4096-long reduction alone), then the 3J real columns are copied out + bias
    P2M_TRY(launch_umma_gemm(y, P->w2_w, B, 64, H, Epilogue(), h, apack, wpack, status, sm_count, s, 3 * J));
    const long long n = (long long)B * 3 * J;
    k_take_cols<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(h, 64, P->w2_b, 3 * J, n, pose3d);
    P2M_LAUNCH_OK();
  } else {
    Epilogue e2;
    e2.bias = P->w2_b;
    P2M_TRY(launch_gemm(y, H, P->w2_w, H, 0, pose3d, 3 * J, B, 3 * J, H, e2, s));
  }
  if (pose_combine != nullptr) {
    const long long n = (long long)B * J;
    k_pose_combine<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(pose2d, pose3d, n, pose_combine);
    P2M_LAUNCH_OK();
  }
  return P2M_OK;
}

}  // extern "C"

// =====================================================================================
// Row f2 of SURVEY.md §8: the steps either side of the model in the reference's callers.
//  * joint regression  joints = J_regressor @ vertices   (lib/core/base.py:131,204; demo/run.py:171)
//  * the demo's input normalisation, demo/run.py:150-158: tight box of the 2-D joints (coord_utils.py:21-39) ->
//    aspect-preserving box of the network input (process_bbox, :42-66) -> affine map into the input_w x input_h
//    patch (aug_utils.py:51-64,140-179 with rot = 0: a uniform scaling that maps the box centre to the patch
//    centre) -> divide by the patch size -> per-pose zero mean / unit std per coordinate.
// =====================================================================================
namespace {
__global__ void __launch_bounds__(256) k_regress_joints(const float* __restrict__ Jr, const float* __restrict__ verts,
                                                        int n_vertex, int chans, float* __restrict__ joints) {
  // one CTA per (joint, mesh); chans <= 4
  const int j = blockIdx.x, n_joint = gridDim.x;
  const long long b = blockIdx.y;
  const float* jr = Jr + (size_t)j * n_vertex;
  const float* vb = verts + b * (long long)n_vertex * chans;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int v = threadIdx.x; v < n_vertex; v += 256) {
    const float w = __ldg(jr + v);
    for (int c = 0; c < chans; ++c) acc[c] = fmaf(w, vb[(long long)v * chans + c], acc[c]);
  }
  __shared__ float red[4][8];
  for (int c = 0; c < 4; ++c) {
    float a = acc[c];
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0) red[c][threadIdx.x >> 5] = a;
  }
  __syncthreads();
  if (threadIdx.x < chans) {
    float a = 0.f;
    for (int w = 0; w < 8; ++w) a += red[threadIdx.x][w];
    joints[(b * n_joint + j) * chans + threadIdx.x] = a;
  }
}

// The box and the affine map of demo/run.py:150-153 for one pose held one joint per lane (all 32 lanes take part;
// lanes >= n_joint pass on = false): get_bbox, process_bbox(aspect_ratio = width / height, scale), then
// j2d_processing into a dst_w x dst_h patch.  Returns the processed box [x, y, w, h] and this lane's joint in patch
// pixels before the reference's cast to float32 (truncated towards zero when truncate is set).
struct PatchPoint {
  float box[4];
  double tx, ty;
};
__device__ __forceinline__ PatchPoint pose_to_patch(float x, float y, bool on, float aspect, float scale, int dst_w_px,
                                                    int dst_h_px, int truncate) {
  float xmin = on ? x : INFINITY, xmax = on ? x : -INFINITY, ymin = on ? y : INFINITY, ymax = on ? y : -INFINITY;
  for (int o = 16; o > 0; o >>= 1) {
    xmin = fminf(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
    xmax = fmaxf(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
    ymin = fminf(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
    ymax = fmaxf(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
  }
  // get_bbox (float32 arithmetic like numpy on the float32 box)
  float bx, by, bw, bh;
  {
    const double xc = ((double)xmin + (double)xmax) / 2.0, w = (double)xmax - (double)xmin;
    const double yc = ((double)ymin + (double)ymax) / 2.0, h = (double)ymax - (double)ymin;
    bx = (float)(xc - 0.5 * w); by = (float)(yc - 0.5 * h); bw = (float)w; bh = (float)h;
  }
  // process_bbox: sanitise (x2 = x + (w - 1)), grow to the aspect ratio width / height, then scale (float32 like numpy
  // on the float32 box; scale 1.0 leaves the box as it is)
  float w = (bx + (bw - 1.f)) - bx, h = (by + (bh - 1.f)) - by;
  const float cx = bx + w / 2.f, cy = by + h / 2.f;
  if (w > aspect * h) h = w / aspect;
  else if (w < aspect * h) w = h * aspect;
  w = w * scale;
  h = h * scale;
  const float x0 = cx - w / 2.f, y0 = cy - h / 2.f;
  PatchPoint p;
  p.box[0] = x0; p.box[1] = y0; p.box[2] = w; p.box[3] = h;
  // get_center_scale + get_affine_transform(rot = 0): three float32 point pairs, solved in double
  const float ccx = x0 + w * 0.5f, ccy = y0 + h * 0.5f;
  const float s1y = ccy + w * -0.5f;                                     // src[1] = centre + (0, -src_w / 2)
  const double dst_w = (double)dst_w_px, dst_h = (double)dst_h_px;
  const float d1y = (float)(dst_h * 0.5) + (float)(dst_w * -0.5);        // dst[1] = (dst_w / 2, dst_h / 2 - dst_w / 2)
  const double sc = ((double)d1y - dst_h * 0.5) / ((double)s1y - (double)ccy);
  p.tx = ((double)x - (double)ccx) * sc + dst_w * 0.5;
  p.ty = ((double)y - (double)ccy) * sc + dst_h * 0.5;
  if (truncate) {  // the reference writes the transformed point back into an INTEGER array (demo/h36m_joint_input.npy
    p.tx = trunc(p.tx);  // is int64): truncation towards zero before astype('float32')
    p.ty = trunc(p.ty);
  }
  return p;
}

// one warp per pose, lane = joint (n_joint <= 32)
__global__ void __launch_bounds__(128) k_normalize_pose2d(const float* __restrict__ px, int batch, int n_joint, int in_h,
                                                          int in_w, int truncate, float* __restrict__ out) {
  const int pose = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (pose >= batch) return;
  const bool on = lane < n_joint;
  const float x = on ? px[((long long)pose * n_joint + lane) * 2 + 0] : 0.f;
  const float y = on ? px[((long long)pose * n_joint + lane) * 2 + 1] : 0.f;
  const PatchPoint p = pose_to_patch(x, y, on, (float)in_w / (float)in_h, 1.f, in_w, in_h, truncate);
  float u = (float)p.tx / (float)in_w, v = (float)p.ty / (float)in_h;
  // per-pose mean / std (population) per coordinate
  float su = on ? u : 0.f, sv = on ? v : 0.f;
  for (int o = 16; o > 0; o >>= 1) {
    su += __shfl_xor_sync(0xffffffffu, su, o);
    sv += __shfl_xor_sync(0xffffffffu, sv, o);
  }
  const float mu = su / n_joint, mv = sv / n_joint;
  float qu = on ? (u - mu) * (u - mu) : 0.f, qv = on ? (v - mv) * (v - mv) : 0.f;
  for (int o = 16; o > 0; o >>= 1) {
    qu += __shfl_xor_sync(0xffffffffu, qu, o);
    qv += __shfl_xor_sync(0xffffffffu, qv, o);
  }
  if (on) {
    out[((long long)pose * n_joint + lane) * 2 + 0] = (u - mu) / sqrtf(qu / n_joint);
    out[((long long)pose * n_joint + lane) * 2 + 1] = (v - mv) / sqrtf(qv / n_joint);
  }
}

// The camera fit's projection target (demo/run.py:150-153 with bbox1 = process_bbox(aspect_ratio, scale)): the joints in
// pixels of the res_w x res_h patch, and the box.  One warp per pose, lane = joint (n_joint <= 32).
__global__ void __launch_bounds__(128) k_crop_pose2d(const float* __restrict__ px, int batch, int n_joint, int res_w,
                                                     int res_h, float aspect, float scale, int truncate,
                                                     float* __restrict__ out, float* __restrict__ out_box) {
  const int pose = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (pose >= batch) return;
  const bool on = lane < n_joint;
  const float x = on ? px[((long long)pose * n_joint + lane) * 2 + 0] : 0.f;
  const float y = on ? px[((long long)pose * n_joint + lane) * 2 + 1] : 0.f;
  const PatchPoint p = pose_to_patch(x, y, on, aspect, scale, res_w, res_h, truncate);
  if (on) {
    out[((long long)pose * n_joint + lane) * 2 + 0] = (float)p.tx;
    out[((long long)pose * n_joint + lane) * 2 + 1] = (float)p.ty;
  }
  if (lane < 4)  // (a select chain, not p.box[lane]: a lane-dependent index would put the box on the stack)
    out_box[(long long)pose * 4 + lane] = lane == 0 ? p.box[0] : (lane == 1 ? p.box[1] : (lane == 2 ? p.box[2] : p.box[3]));
}

// demo/run.py:160-189: the weak-perspective camera of lib/models/project_net.py,
//   out = (p[:, :2] + c[1:]) * c[0] * R + R,   R = crop_size / 2,
// fitted to the target by `iters` steps of mean-L1 loss + torch.optim.Adam (defaults, lr 0.1 / 0.05 / 0.001 after steps
// 501 / 1001).  One warp per person, lane = joint: the camera, the Adam moments and the step count live in registers
// for the whole fit.  With s = sign(out - tgt) (sign(0) = 0, torch's abs backward) and N = 2 n_joint,
//   dL/dc1 = R c0 / N * sum_j s_x,   dL/dc2 = R c0 / N * sum_j s_y,   dL/dc0 = R / N * sum_j (s_x a_x + s_y a_y)
// with a = p + c[1:]: the first two are counts of signs (ballot + popc), the third one float warp reduction.  The
// arithmetic is written op by op in round-to-nearest (no FMA contraction) in the order of the reference's fp32 torch
// ops; Adam's bias corrections are computed in double as torch does on the host.
__device__ __forceinline__ float warp_sum(float v) {
  // xor butterfly: every lane ends with the same bits (each level adds the same two values, a + b == b + a)
  for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, float step, float bc2_sqrt) {
  m = __fadd_rn(m, __fmul_rn(0.1f, __fsub_rn(g, m)));                       // exp_avg.lerp_(grad, 1 - beta1)
  v = __fadd_rn(__fmul_rn(v, 0.999f), __fmul_rn(__fmul_rn(0.001f, g), g));  // exp_avg_sq.mul_(b2).addcmul_(g, g, 1 - b2)
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), 1e-8f);
  p = __fadd_rn(p, __fdiv_rn(__fmul_rn(-step, m), denom));                  // param.addcdiv_(m, denom, -step_size)
}

__global__ void __launch_bounds__(128) k_fit_camera(const float* __restrict__ j3d, const float* __restrict__ tgt,
                                                    const float* __restrict__ cam_init, int batch, int n_joint,
                                                    int stride, float R, int iters, float* __restrict__ cam_out,
                                                    float* __restrict__ loss_out) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= batch) return;
  const bool on = lane < n_joint;
  const long long jb = (long long)b * n_joint + lane;
  const float px = on ? j3d[jb * stride + 0] : 0.f, py = on ? j3d[jb * stride + 1] : 0.f;
  const float qx = on ? tgt[jb * 2 + 0] : 0.f, qy = on ? tgt[jb * 2 + 1] : 0.f;
  float c0 = cam_init[b * 3 + 0], c1 = cam_init[b * 3 + 1], c2 = cam_init[b * 3 + 2];
  float m0 = 0.f, m1 = 0.f, m2 = 0.f, v0 = 0.f, v1 = 0.f, v2 = 0.f;
  const float gs = __fmul_rn(__fdiv_rn(1.f, (float)(2 * n_joint)), R);  // mean backward (1 / N), then the "* R"
  for (int t = 1; t <= iters; ++t) {
    const float ax = __fadd_rn(px, c1), ay = __fadd_rn(py, c2);
    const float rx = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(ax, c0), R), R), qx);
    const float ry = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(ay, c0), R), R), qy);
    const int sx = __popc(__ballot_sync(0xffffffffu, on && rx > 0.f)) - __popc(__ballot_sync(0xffffffffu, on && rx < 0.f));
    const int sy = __popc(__ballot_sync(0xffffffffu, on && ry > 0.f)) - __popc(__ballot_sync(0xffffffffu, on && ry < 0.f));
    float sa = 0.f;
    if (on) {
      sa = rx > 0.f ? ax : (rx < 0.f ? -ax : 0.f);
      sa = __fadd_rn(sa, ry > 0.f ? ay : (ry < 0.f ? -ay : 0.f));
    }
    const float g0 = __fmul_rn(gs, warp_sum(sa));
    const float gc = __fmul_rn(gs, c0);
    const float g1 = __fmul_rn((float)sx, gc), g2 = __fmul_rn((float)sy, gc);
    // lr schedule of run.py:181-186 (the change after loop index 500 / 1000 applies from the next step on)
    const double lr = t <= 501 ? 0.1 : (t <= 1001 ? 0.05 : 0.001);
    const float step = (float)(lr / (1.0 - pow(0.9, (double)t)));
    const float bc2_sqrt = (float)sqrt(1.0 - pow(0.999, (double)t));
    adam_update(c0, m0, v0, g0, step, bc2_sqrt);
    adam_update(c1, m1, v1, g1, step, bc2_sqrt);
    adam_update(c2, m2, v2, g2, step, bc2_sqrt);
  }
  // L1 loss of the final camera (nn.L1Loss: mean over the n_joint x 2 residuals)
  const float ax = __fadd_rn(px, c1), ay = __fadd_rn(py, c2);
  const float rx = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(ax, c0), R), R), qx);
  const float ry = __fsub_rn(__fadd_rn(__fmul_rn(__fmul_rn(ay, c0), R), R), qy);
  const float l = warp_sum(on ? __fadd_rn(fabsf(rx), fabsf(ry)) : 0.f);
  if (lane == 0) {
    cam_out[b * 3 + 0] = c0;
    cam_out[b * 3 + 1] = c1;
    cam_out[b * 3 + 2] = c2;
    loss_out[b] = __fdiv_rn(l, (float)(2 * n_joint));
  }
}
}  // namespace

extern "C" {

int p2m_regress_joints(const float* joint_regressor, const float* vertices, float* joints, int batch, int n_joint,
                       int n_vertex, int chans, p2m_stream_t stream) {
  if (!joint_regressor || !vertices || !joints || batch <= 0 || n_joint <= 0 || n_vertex <= 0 || chans <= 0 || chans > 4 ||
      batch > 65535) {
    set_error("regress_joints: bad argument");
    return P2M_ERR_INVALID;
  }
  k_regress_joints<<<dim3(n_joint, batch), 256, 0, static_cast<cudaStream_t>(stream)>>>(joint_regressor, vertices,
                                                                                       n_vertex, chans, joints);
  P2M_LAUNCH_OK();
  return P2M_OK;
}

int p2m_normalize_pose2d(const float* joints_px, float* pose2d, int batch, int n_joint, int input_h, int input_w,
                         int truncate_like_int_input, p2m_stream_t stream) {
  if (!joints_px || !pose2d || batch <= 0 || n_joint <= 0 || n_joint > 32 || input_h <= 0 || input_w <= 0) {
    set_error("normalize_pose2d: bad argument (at most 32 joints)");
    return P2M_ERR_INVALID;
  }
  k_normalize_pose2d<<<(batch + 3) / 4, 128, 0, static_cast<cudaStream_t>(stream)>>>(joints_px, batch, n_joint, input_h,
                                                                                   input_w, truncate_like_int_input, pose2d);
  P2M_LAUNCH_OK();
  return P2M_OK;
}

int p2m_crop_pose2d(const float* joints_px, float* out_px, float* out_bbox, int batch, int n_joint, int res_w, int res_h,
                    float aspect_ratio, float scale, int truncate_like_int_input, p2m_stream_t stream) {
  if (!joints_px || !out_px || !out_bbox || batch <= 0 || n_joint <= 0 || n_joint > 32 || res_w <= 0 || res_h <= 0 ||
      !(aspect_ratio > 0.f) || !(scale > 0.f)) {
    set_error("crop_pose2d: bad argument (null pointer, at most 32 joints, positive patch size / aspect ratio / scale)");
    return P2M_ERR_INVALID;
  }
  k_crop_pose2d<<<(batch + 3) / 4, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      joints_px, batch, n_joint, res_w, res_h, aspect_ratio, scale, truncate_like_int_input, out_px, out_bbox);
  P2M_LAUNCH_OK();
  return P2M_OK;
}

int p2m_fit_camera(const float* joints3d, const float* target_px, const float* cam_init, float* cam_out, float* loss_out,
                   int batch, int n_joint, int joint_stride, double crop_size, int iters, p2m_stream_t stream) {
  if (!joints3d || !target_px || !cam_init || !cam_out || !loss_out) {
    set_error("fit_camera: null pointer");
    return P2M_ERR_INVALID;
  }
  if (batch <= 0 || n_joint <= 0 || n_joint > 32) {
    set_error("fit_camera: need batch >= 1 and 1 <= n_joint <= 32 (got batch " + std::to_string(batch) + ", n_joint " +
              std::to_string(n_joint) + ")");
    return P2M_ERR_INVALID;
  }
  if (joint_stride < 2 || iters < 1 || !(crop_size > 0.0)) {
    set_error("fit_camera: need joint_stride >= 2, iters >= 1 and crop_size > 0 (got " + std::to_string(joint_stride) +
              ", " + std::to_string(iters) + ", " + std::to_string(crop_size) + ")");
    return P2M_ERR_INVALID;
  }
  k_fit_camera<<<(batch + 3) / 4, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      joints3d, target_px, cam_init, batch, n_joint, joint_stride, (float)(crop_size / 2.0), iters, cam_out, loss_out);
  P2M_LAUNCH_OK();
  return P2M_OK;
}

}  // extern "C"

// =====================================================================================
// Row f3 of SURVEY.md §8: the mesh losses of lib/core/loss.py on the GPU, forward and backward in one pass.
//   NormalVectorLoss (:62-87)  mean over (B, 3 Nf) of |<normalize(edge_i(out)), normal(gt)>|
//   EdgeLengthLoss   (:90-114) mean over (B, 3 Nf) of | |edge_i(out)| - |edge_i(gt)| |
//   CoordLoss        (:10-23)  mean |pred * valid - target * valid|
// The reference rebuilds a LongTensor of the faces on the device in EVERY call (:68, :97) and materialises ~20
// [B, Nf, 3] temporaries; here one thread handles one (mesh, face): 18 loads, the two loss terms, and — when
// gradients are wanted — 9 atomic adds into d(coord_out).  F.normalize semantics: v / max(|v|, 1e-12).
// =====================================================================================
namespace {
struct V3 {
  float x, y, z;
};
__device__ __forceinline__ V3 sub3(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ float dot3(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 scale3(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
__device__ __forceinline__ V3 normalize3(V3 a, float* len) {
  const float n = sqrtf(dot3(a, a));
  *len = n;
  return scale3(a, 1.f / fmaxf(n, 1e-12f));
}
__device__ __forceinline__ V3 ld3(const float* p) { return V3{p[0], p[1], p[2]}; }
__device__ __forceinline__ void atomic_add3(float* p, V3 g) {
  atomicAdd(p + 0, g.x);
  atomicAdd(p + 1, g.y);
  atomicAdd(p + 2, g.z);
}

// sums[0] += sum of the 3 normal terms, sums[1] += sum of the 3 edge terms (fp64); grad (optional, zeroed by the
// caller) += g_normal * d(normal sum)/d(out) + g_edge * d(edge sum)/d(out) with g_* already divided by 3 B Nf.
__global__ void __launch_bounds__(256) k_mesh_losses(const float* __restrict__ out, const float* __restrict__ gt,
                                                     const int* __restrict__ faces, int n_face, int n_vertex, int batch,
                                                     const float* __restrict__ g_scale, double* __restrict__ sums,
                                                     float* __restrict__ grad) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float ln = 0.f, le = 0.f;
  if (idx < (long long)batch * n_face) {
    const int f = (int)(idx % n_face);
    const long long b = idx / n_face;
    const int i0 = faces[3 * f], i1 = faces[3 * f + 1], i2 = faces[3 * f + 2];
    const float* ob = out + b * (long long)n_vertex * 3;
    const float* gb = gt + b * (long long)n_vertex * 3;
    const V3 o0 = ld3(ob + 3 * i0), o1 = ld3(ob + 3 * i1), o2 = ld3(ob + 3 * i2);
    const V3 t0 = ld3(gb + 3 * i0), t1 = ld3(gb + 3 * i1), t2 = ld3(gb + 3 * i2);
    // ---- normal-vector term
    float l1, l2, l3, lg;
    const V3 e1 = sub3(o1, o0), e2 = sub3(o2, o0), e3 = sub3(o2, o1);
    const V3 u1 = normalize3(e1, &l1), u2 = normalize3(e2, &l2), u3 = normalize3(e3, &l3);
    const V3 a = normalize3(sub3(t1, t0), &lg), c = normalize3(sub3(t2, t0), &lg);
    const V3 n = normalize3(V3{a.y * c.z - a.z * c.y, a.z * c.x - a.x * c.z, a.x * c.y - a.y * c.x}, &lg);
    const float c1 = dot3(u1, n), c2 = dot3(u2, n), c3 = dot3(u3, n);
    ln = fabsf(c1) + fabsf(c2) + fabsf(c3);
    // ---- edge-length term (reference edge order: (0,1), (0,2), (1,2))
    const float d1 = l1, d2 = l2, d3 = l3;  // |o0-o1|, |o0-o2|, |o1-o2|
    float q1, q2, q3;
    normalize3(sub3(t0, t1), &q1);
    normalize3(sub3(t0, t2), &q2);
    normalize3(sub3(t1, t2), &q3);
    const float r1 = d1 - q1, r2 = d2 - q2, r3 = d3 - q3;
    le = fabsf(r1) + fabsf(r2) + fabsf(r3);
    if (grad != nullptr) {
      const float gn = g_scale[0], ge = g_scale[1];
      float* gr = grad + b * (long long)n_vertex * 3;
      // d|<u, n>| / de = sign(<u,n>) (n - u <u,n>) / |e|   (|e| > eps); sign(0) = 0 like torch.abs
      auto dcos = [&](V3 u, float cs, float len) {
        const float sg = (cs > 0.f) - (cs < 0.f);
        const float inv = (len > 1e-12f) ? sg / len : 0.f;
        return scale3(sub3(n, scale3(u, cs)), inv * gn);
      };
      // d| |e| - q | / de = sign(|e| - q) e / |e|
      auto dlen = [&](V3 u, float r, float len) {
        const float sg = (r > 0.f) - (r < 0.f);
        return scale3(u, (len > 0.f) ? sg * ge : 0.f);
      };
      V3 g1 = dcos(u1, c1, l1), g2 = dcos(u2, c2, l2), g3 = dcos(u3, c3, l3);       // w.r.t. e1, e2, e3
      const V3 h1 = dlen(u1, r1, l1), h2 = dlen(u2, r2, l2), h3 = dlen(u3, r3, l3);  // same edges (sign-symmetric)
      g1 = V3{g1.x + h1.x, g1.y + h1.y, g1.z + h1.z};
      g2 = V3{g2.x + h2.x, g2.y + h2.y, g2.z + h2.z};
      g3 = V3{g3.x + h3.x, g3.y + h3.y, g3.z + h3.z};
      // e1 = o1 - o0, e2 = o2 - o0, e3 = o2 - o1
      atomic_add3(gr + 3 * i0, V3{-g1.x - g2.x, -g1.y - g2.y, -g1.z - g2.z});
      atomic_add3(gr + 3 * i1, V3{g1.x - g3.x, g1.y - g3.y, g1.z - g3.z});
      atomic_add3(gr + 3 * i2, V3{g2.x + g3.x, g2.y + g3.y, g2.z + g3.z});
    }
  }
  __shared__ float red[2][8];
  for (int o = 16; o > 0; o >>= 1) {
    ln += __shfl_xor_sync(0xffffffffu, ln, o);
    le += __shfl_xor_sync(0xffffffffu, le, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = ln;
    red[1][threadIdx.x >> 5] = le;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[threadIdx.x][w];
    atomicAdd(sums + threadIdx.x, s);
  }
}

// CoordLoss: sums[0] += sum |p v - t v|; grad (optional) = g * sign(p v - t v) * v
__global__ void __launch_bounds__(256) k_coord_loss(const float* __restrict__ pred, const float* __restrict__ target,
                                                    const float* __restrict__ valid, long long n,
                                                    const float* __restrict__ g_scale, double* __restrict__ sums,
                                                    float* __restrict__ grad) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float l = 0.f;
  if (i < n) {
    const float v = valid ? valid[i] : 1.f;
    const float d = pred[i] * v - target[i] * v;
    l = fabsf(d);
    if (grad != nullptr) grad[i] = g_scale[0] * (float)((d > 0.f) - (d < 0.f)) * v;
  }
  __shared__ float red[8];
  for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = l;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[w];
    atomicAdd(sums, s);
  }
}
}  // namespace

extern "C" {

int p2m_mesh_losses(const float* coord_out, const float* coord_gt, const int32_t* faces, int batch, int n_vertex,
                    int n_face, const float* grad_scale, double* sums, float* grad_out, p2m_stream_t stream) {
  if (!coord_out || !coord_gt || !faces || !sums || batch <= 0 || n_vertex <= 0 || n_face <= 0 ||
      (grad_out != nullptr && grad_scale == nullptr)) {
    set_error("mesh_losses: bad argument");
    return P2M_ERR_INVALID;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  P2M_CUDA_OK(cudaMemsetAsync(sums, 0, 2 * sizeof(double), s));
  if (grad_out) P2M_CUDA_OK(cudaMemsetAsync(grad_out, 0, sizeof(float) * 3 * (size_t)batch * n_vertex, s));
  const long long n = (long long)batch * n_face;
  k_mesh_losses<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(coord_out, coord_gt, faces, n_face, n_vertex, batch, grad_scale,
                                                            sums, grad_out);
  P2M_LAUNCH_OK();
  return P2M_OK;
}

int p2m_coord_loss(const float* pred, const float* target, const float* valid, int64_t n, const float* grad_scale,
                   double* sum, float* grad_out, p2m_stream_t stream) {
  if (!pred || !target || !sum || n <= 0 || (grad_out != nullptr && grad_scale == nullptr)) {
    set_error("coord_loss: bad argument");
    return P2M_ERR_INVALID;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  P2M_CUDA_OK(cudaMemsetAsync(sum, 0, sizeof(double), s));
  k_coord_loss<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(pred, target, valid, n, grad_scale, sum, grad_out);
  P2M_LAUNCH_OK();
  return P2M_OK;
}

}  // extern "C"
