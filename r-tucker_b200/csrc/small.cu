// (c) The N-independent part of one Riemannian optimiser step, in fp64 on the device.
//
// Restates, at rank r (no rank-2r construct, no autodiff), what the reference obtains from
// tucker_riemopt 1.0.1: the (S_(i)S_(i)^T)^-1 factors and the gauge projection of `grad`
// (call sites src/model/asymmetric/optim.py:89, symmetric/optim.py:83), `TangentVector.norm`
// (asymmetric/optim.py:90), `project` (asymmetric/optim.py:86) and the core part of
// `construct().round(rank)` (asymmetric/optim.py:108) -- the latter as the structured HOSVD of
// SURVEY.md App. A.5 (Cholesky of the W_i Grams, block-structured rank-2r core, dominant invariant
// subspaces of the unfolding Grams, subspace.cu) instead of QR(N x 2r) + SVD(2r_i x prod 2r_j).
//
// Everything here costs O(poly(r)) and is replicated on every GPU of an entity-sharded run.
#include "small_kernels.cuh"
#include "small_exec.cuh"

#include <algorithm>
#include <vector>

namespace {
using namespace rt::small;
using rt::align_up;
using rt::cdiv;

constexpr int kNumT = 8;          // core-sized fp64 temporaries
constexpr int kMinDotSlots = 2048;
// Arena of the executor's split-K partial sums: 592 tiles of 64 x 64 doubles.  Ctx::gemm_any splits a GEMM over K only
// when its partials fit here, so this size fixes the order of the sums: changing it changes results in the last bits.
constexpr size_t kPartialArenaBytes = (size_t)592 * 64 * 64 * sizeof(double);

struct Layout {
  int r[3];
  int B;
  int64_t c;  // r0*r1*r2
  size_t C64, Gm[3], Ainv[3], coresq, Tn[kNumT], KC[3], Nn[3], Vf[3], GL[3], GLinv[3], Gs[3],
      tmpM[3], tmpK[3], sub[3], sub_shared, exec_bar, gemm_partial, gram_ws, dot_partial, scal, total;
  int dot_slots;  // doubles at dot_partial: one per kEwChunk elements of the dots recorded between two flushes
};

Layout make_layout(int r0, int r1, int r2, int B) {
  Layout L;
  L.r[0] = r0; L.r[1] = r1; L.r[2] = r2; L.B = B;
  L.c = (int64_t)r0 * r1 * r2;
  rt::WsArena ws;
  auto take = [&](size_t doubles) { return ws.take(doubles * sizeof(double)); };
  L.C64 = take(L.c);
  for (int i = 0; i < 3; ++i) { L.Gm[i] = take((size_t)L.r[i] * L.r[i]); L.Ainv[i] = take((size_t)L.r[i] * L.r[i]); }
  L.coresq = take(4);
  for (int t = 0; t < kNumT; ++t) L.Tn[t] = take(L.c);
  for (int i = 0; i < 3; ++i) {
    const size_t r = L.r[i];
    L.KC[i] = take(2 * r * r);
    L.Nn[i] = take(4 * r * r);
    L.Vf[i] = take(4 * r * r);
    L.GL[i] = take(r * r);
    L.GLinv[i] = take(r * r);
    L.Gs[i] = take(r * r);
    L.tmpM[i] = take(2 * r * r);
    L.tmpK[i] = take(2 * r * r);
    L.sub[i] = ws.take(rt::subspace_ws_bytes(2 * (int)r, (int)r));
  }
  L.sub_shared = ws.take(rt::subspace_shared_ws_bytes());
  L.exec_bar = take(32);        // two grid-barrier counters, 128 bytes apart (Ctx::flush)
  L.gemm_partial = take(kPartialArenaBytes / sizeof(double));
  int rmax = r0 > r1 ? r0 : r1; rmax = rmax > r2 ? rmax : r2;
  L.gram_ws = ws.take(rt_gram_ws_bytes(B > 0 ? B : 1, rmax, rmax));
  // The largest dots (rt_small_norm) are one over the core and one over each r_i x r_i Gram, recorded together;
  // every partial of one dot must fit, or its two-stage sum would write past the slot.
  auto chunks = [](int64_t n) { return (n + kEwChunk - 1) / kEwChunk; };
  int64_t slots = chunks(L.c);
  for (int i = 0; i < 3; ++i) slots += chunks((int64_t)L.r[i] * L.r[i]);
  L.dot_slots = (int)std::max<int64_t>(kMinDotSlots, slots);
  L.dot_partial = take((size_t)L.dot_slots);
  L.scal = take(16);
  L.total = ws.o;
  return L;
}

// ---- recording context: operations are RECORDED with the byte ranges they touch, scheduled into dependency
// levels and executed by one persistent launch per flush() (small_exec.cuh) ------------------------------------------
struct Range { const char* lo; const char* hi; };
struct Rec { Op op; Range rd[4]; int nrd; Range wr[4]; int nwr; };

// C[m,n] = alpha * sum_{k1<K1,k2<K2} A[m,(k1,k2)] B[(k1,k2),n] + beta * C[m,n]      (batched): what Ctx::mode_prod and
// Ctx::unfold_gram hand to Ctx::gemm
template <typename T>
struct GemmT {
  const T* A; const T* B; T* C;
  int m, n, K1, K2;
  int64_t a_m, a_k1, a_k2;
  int64_t b_k1, b_k2, b_n;
  int64_t c_m, c_n;
  int batch; int64_t a_b, b_b, c_b;
  double alpha, beta;
  int sym;                  // C is symmetric (A = B with equal strides): compute the upper triangle of tiles only
};

template <typename T> struct DT;
template <> struct DT<float> { static constexpr int v = DT_F32; };
template <> struct DT<double> { static constexpr int v = DT_F64; };
static inline size_t dsize(int t) { return t == DT_F64 ? 8 : 4; }

enum class Launch { kCooperative, kAfterPrimary };

struct Ctx {
  Layout L;
  char* base;
  cudaStream_t s;
  int err = 0;
  std::vector<Rec> recs;
  size_t partial_off = 0;
  int dot_off = 0;
  double* p(size_t off) const { return (double*)(base + off); }
  double* T(int t) const { return p(L.Tn[t]); }
  int r(int i) const { return L.r[i]; }

  static Range range(const void* ptr, size_t bytes) { return Range{(const char*)ptr, (const char*)ptr + bytes}; }
  static bool overlap(const Range& a, const Range& b) { return a.lo < b.hi && b.lo < a.hi; }

  void push(Rec& rec) {
    if (err) return;
    if ((int)recs.size() >= kMaxOps) flush();
    // level = 1 + the deepest earlier operation this one conflicts with (RAW, WAW, WAR on byte ranges)
    int level = 0;
    for (const Rec& q : recs) {
      bool c = false;
      for (int i = 0; i < q.nwr && !c; ++i) {
        for (int j = 0; j < rec.nrd && !c; ++j) c = overlap(q.wr[i], rec.rd[j]);
        for (int j = 0; j < rec.nwr && !c; ++j) c = overlap(q.wr[i], rec.wr[j]);
      }
      for (int i = 0; i < q.nrd && !c; ++i)
        for (int j = 0; j < rec.nwr && !c; ++j) c = overlap(q.rd[i], rec.wr[j]);
      if (c && q.op.level + 1 > level) level = q.op.level + 1;
    }
    rec.op.level = level;
    recs.push_back(rec);
  }

  // Execute what has been recorded as one cooperative launch of `ctas` CTAs (0: kExecCtasPerSm per SM); direct
  // launches may follow on the stream.  Launch::kAfterPrimary makes the program the programmatic dependent of the
  // kernel enqueued just before it: it may start while that kernel runs, on the SMs that kernel leaves free, and it
  // ends only after that kernel has completed (pdl_wait).  No memset may come between the two launches, so such a
  // program counts on the second counter of exec_bar instead: every cooperative flush zeroes both, and only a
  // dependent program advances the second.
  void flush(int ctas = 0, Launch mode = Launch::kCooperative) {
    if (err || recs.empty()) { recs.clear(); return; }
    std::stable_sort(recs.begin(), recs.end(), [](const Rec& a, const Rec& b) { return a.op.level < b.op.level; });
    static Program prog;     // host staging of the parameter block (copied by the launch)
    const bool dependent = mode == Launch::kAfterPrimary;
    prog.nops = (int)recs.size();
    prog.bar = reinterpret_cast<unsigned int*>(base + L.exec_bar) + (dependent ? 32 : 0);
    for (int i = 0; i < prog.nops; ++i) prog.ops[i] = recs[i].op;
    recs.clear();
    partial_off = 0;
    dot_off = 0;
    const size_t smem = sizeof(double) * kExecWarps * XT * XLD;
    if ((!dependent && cudaMemsetAsync(base + L.exec_bar, 0, 256, s) != cudaSuccess) ||
        cudaFuncSetAttribute(small_exec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
            cudaSuccess) {
      err = 1; return;
    }
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ctas > 0 ? ctas : kExecCtasPerSm * rt::sm_count());
    cfg.blockDim = dim3(kExecThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cfg.attrs = attr;
    cfg.numAttrs = dependent ? 2 : 1;
    void* args[] = {(void*)&prog};
    if (cudaLaunchKernelExC(&cfg, (const void*)small_exec_kernel, args) != cudaSuccess) err = 1;
    ++rt::g_launches;
  }

  // C (tc) [m, n] = alpha * (alpha_dev ? *alpha_dev : 1) * sum_{k1, k2} A (ta) B (tb) + beta * C, batched; element strides
  void gemm_any(const void* A, int ta, const void* B, int tb, void* C, int tc, int m, int n, int K1, int K2,
                int64_t a_m, int64_t a_k1, int64_t a_k2, int64_t b_k1, int64_t b_k2, int64_t b_n, int64_t c_m,
                int64_t c_n, int batch, int64_t a_b, int64_t b_b, int64_t c_b, double alpha, double beta,
                const double* alpha_dev = nullptr, bool sym = false) {
    if (err || m <= 0 || n <= 0) return;
    if (m != n || batch != 1) sym = false;
    Rec rec{};
    GemmPart& g = rec.op.g;
    rec.op.kind = OP_GEMM;
    g.A = A; g.B = B; g.C = C; g.ta = ta; g.tb = tb; g.tc = tc;
    g.m = m; g.n = n; g.K1 = K1; g.K2 = K2;
    g.a_m = a_m; g.a_k1 = a_k1; g.a_k2 = a_k2; g.b_k1 = b_k1; g.b_k2 = b_k2; g.b_n = b_n; g.c_m = c_m; g.c_n = c_n;
    g.batch = batch; g.a_b = a_b; g.b_b = b_b; g.c_b = c_b;
    g.alpha = alpha; g.beta = beta; g.alpha_dev = alpha_dev;
    g.tiles_m = cdiv(m, XT); g.tiles_n = cdiv(n, XT);
    g.sym = sym ? 1 : 0;
    const int tiles = sym ? g.tiles_n * (g.tiles_n + 1) / 2 : batch * g.tiles_m * g.tiles_n;
    const int S = K1 * cdiv(K2, 4);
    g.ksplit = 1; g.steps_per_split = S > 0 ? S : 1; g.partial = nullptr;
    if (tiles < 120 && S >= 32) {
      int ks = cdiv(160, tiles);
      if (ks > S / 16) ks = S / 16;
      if (ks > 64) ks = 64;
      if (ks > 1) {
        const int sps = cdiv(cdiv(S, ks), kExecWarps) * kExecWarps;
        ks = cdiv(S, sps);
        const size_t bytes = align_up((size_t)ks * batch * m * n * sizeof(double), 256);
        if (ks > 1 && bytes <= kPartialArenaBytes) {
          if (partial_off + bytes > kPartialArenaBytes) partial_off = 0;   // wrap: the hazard tracking orders the reuse
          g.partial = reinterpret_cast<double*>(base + L.gemm_partial + partial_off);
          partial_off += bytes;
          g.ksplit = ks; g.steps_per_split = sps;
        }
      }
    }
    rt::g_small_flops += (sym ? 1.0 : 2.0) * (double)batch * m * n * (double)K1 * K2;   // algorithmic (a Gram: half)
    rec.op.units = tiles * g.ksplit;
    g.thin = (m <= kThinM && K1 == 1 && K2 <= kThinK && batch == 1 && g.ksplit == 1 && n >= 4 * kThinCols) ? 1 : 0;
    if (g.thin) { rec.op.units = cdiv(n, kThinCols); g.sym = 0; }
    auto ext = [](int64_t a, int64_t b, int64_t c, int64_t d) { return (size_t)(a + b + c + d + 1); };
    const size_t ea = ext((int64_t)(m - 1) * a_m, (int64_t)(K1 - 1) * a_k1, (int64_t)(K2 - 1) * a_k2, (int64_t)(batch - 1) * a_b);
    const size_t eb = ext((int64_t)(n - 1) * b_n, (int64_t)(K1 - 1) * b_k1, (int64_t)(K2 - 1) * b_k2, (int64_t)(batch - 1) * b_b);
    const size_t ec = ext((int64_t)(m - 1) * c_m, (int64_t)(n - 1) * c_n, 0, (int64_t)(batch - 1) * c_b);
    rec.rd[rec.nrd++] = range(A, ea * dsize(ta));
    rec.rd[rec.nrd++] = range(B, eb * dsize(tb));
    if (alpha_dev) rec.rd[rec.nrd++] = range(alpha_dev, 8);
    if (g.ksplit > 1) {
      rec.wr[rec.nwr++] = range(g.partial, (size_t)g.ksplit * batch * m * n * sizeof(double));
      push(rec);
      Rec red{};
      red.op.kind = OP_REDUCE;
      red.op.g = g;
      red.op.units = cdiv(batch * m * n, kReduceChunk);
      red.rd[red.nrd++] = range(g.partial, (size_t)g.ksplit * batch * m * n * sizeof(double));
      if (alpha_dev) red.rd[red.nrd++] = range(alpha_dev, 8);
      if (beta != 0.0) red.rd[red.nrd++] = range(C, ec * dsize(tc));
      red.wr[red.nwr++] = range(C, ec * dsize(tc));
      push(red);
    } else {
      if (beta != 0.0) rec.rd[rec.nrd++] = range(C, ec * dsize(tc));
      rec.wr[rec.nwr++] = range(C, ec * dsize(tc));
      push(rec);
    }
  }

  template <typename T>
  void gemm(const GemmT<T>& g) {
    gemm_any(g.A, DT<T>::v, g.B, DT<T>::v, g.C, DT<T>::v, g.m, g.n, g.K1, g.K2, g.a_m, g.a_k1, g.a_k2, g.b_k1, g.b_k2,
             g.b_n, g.c_m, g.c_n, g.batch, g.a_b, g.b_b, g.c_b, g.alpha, g.beta, nullptr, g.sym != 0);
  }

  // Y = alpha * (X x_mode M) + beta * Y.  M is (mo x mi) with strides (sm_o, sm_i);
  // X has dims d[] with d[mode] == mi; Y has the same dims except d[mode] -> mo.
  template <typename T>
  void mode_prod(int mode, const T* M, int64_t sm_o, int64_t sm_i, int mo, int mi,
                 const T* X, const int d[3], T* Y, double alpha, double beta) {
    GemmT<T> g{};
    g.alpha = alpha; g.beta = beta; g.batch = 1;
    if (mode == 0) {
      const int64_t rest = (int64_t)d[1] * d[2];
      g.A = M; g.B = X; g.C = Y; g.m = mo; g.n = (int)rest; g.K1 = 1; g.K2 = mi;
      g.a_m = sm_o; g.a_k1 = 0; g.a_k2 = sm_i; g.b_k1 = 0; g.b_k2 = rest; g.b_n = 1;
      g.c_m = rest; g.c_n = 1;
    } else if (mode == 1) {
      g.A = M; g.B = X; g.C = Y; g.m = mo; g.n = d[2]; g.K1 = 1; g.K2 = mi;
      g.a_m = sm_o; g.a_k1 = 0; g.a_k2 = sm_i; g.b_k1 = 0; g.b_k2 = d[2]; g.b_n = 1;
      g.c_m = d[2]; g.c_n = 1;
      g.batch = d[0]; g.a_b = 0; g.b_b = (int64_t)mi * d[2]; g.c_b = (int64_t)mo * d[2];
    } else {
      g.A = X; g.B = M; g.C = Y; g.m = d[0] * d[1]; g.n = mo; g.K1 = 1; g.K2 = mi;
      g.a_m = mi; g.a_k1 = 0; g.a_k2 = 1; g.b_k1 = 0; g.b_k2 = sm_i; g.b_n = sm_o;
      g.c_m = mo; g.c_n = 1;
    }
    gemm(g);
  }

  // out[mx, my] (row stride ldo) = alpha * X_(mode) Y_(mode)^T + beta * out.
  // X dims dx[], Y dims equal to dx except dy_mode in the contracted-free mode.
  template <typename T>
  void unfold_gram(int mode, const T* X, const int dx[3], const T* Y, int my, T* out,
                   int64_t ldo, double alpha, double beta) {
    GemmT<T> g{};
    g.alpha = alpha; g.beta = beta; g.batch = 1;
    g.A = X; g.B = Y; g.C = out; g.m = dx[mode]; g.n = my; g.c_m = ldo; g.c_n = 1;
    g.sym = (X == Y && my == dx[mode]) ? 1 : 0;      // X_(mode) X_(mode)^T: symmetric, half the tiles
    if (mode == 0) {
      const int64_t rest = (int64_t)dx[1] * dx[2];
      g.K1 = 1; g.K2 = (int)rest;
      g.a_m = rest; g.a_k1 = 0; g.a_k2 = 1; g.b_k1 = 0; g.b_k2 = 1; g.b_n = rest;
    } else if (mode == 1) {
      g.K1 = dx[0]; g.K2 = dx[2];
      g.a_m = dx[2]; g.a_k1 = (int64_t)dx[1] * dx[2]; g.a_k2 = 1;
      g.b_n = dx[2]; g.b_k1 = (int64_t)my * dx[2]; g.b_k2 = 1;
    } else {
      g.K1 = 1; g.K2 = dx[0] * dx[1];
      g.a_m = 1; g.a_k1 = 0; g.a_k2 = dx[2]; g.b_k1 = 0; g.b_k2 = my; g.b_n = 1;
    }
    gemm(g);
  }

  // plain C[m,n] = alpha * A[m,k] B[k,n] + beta*C with row-major leading dims
  void matmul(const double* A, int64_t lda, bool ta, const double* B, int64_t ldb, bool tb, double* C,
              int64_t ldc, int m, int n, int k, double alpha, double beta, const double* alpha_dev = nullptr) {
    gemm_any(A, DT_F64, B, DT_F64, C, DT_F64, m, n, 1, k, ta ? 1 : lda, 0, ta ? lda : 1, 0, tb ? 1 : ldb, tb ? ldb : 1,
             ldc, 1, 1, 0, 0, 0, alpha, beta, alpha_dev);
  }

  float* Tf(int t) const { return reinterpret_cast<float*>(T(t)); }   // the same temporaries viewed as fp32

  void ew(int kind, const void* x, int tx, size_t xbytes, const void* y, size_t ybytes, void* z, int tz, size_t zbytes,
          int64_t count, double s0, const double* d0, double s1, const double* d1, int64_t p0 = 0, int64_t p1 = 0,
          int64_t p2 = 0, int64_t p3 = 0, bool reads_z = false, size_t d0_bytes = 8) {
    if (err || count <= 0) return;
    Rec rec{};
    rec.op.kind = OP_EW; rec.op.ew = kind;
    EwPart& e = rec.op.e;
    e.x = x; e.y = y; e.z = z; e.tx = tx; e.tz = tz; e.count = count; e.s0 = s0; e.s1 = s1; e.d0 = d0; e.d1 = d1;
    e.p0 = p0; e.p1 = p1; e.p2 = p2; e.p3 = p3;
    rec.op.units = kind == EW_NORM_FINISH ? 1 : (int)((count + kEwChunk - 1) / kEwChunk);
    if (x) rec.rd[rec.nrd++] = range(x, xbytes);
    if (y) rec.rd[rec.nrd++] = range(y, ybytes);
    if (d0) rec.rd[rec.nrd++] = range(d0, d0_bytes);
    if (d1) rec.rd[rec.nrd++] = range(d1, 8);
    if (reads_z && rec.nrd < 4) rec.rd[rec.nrd++] = range(z, zbytes);
    rec.wr[rec.nwr++] = range(z, zbytes);
    push(rec);
  }
  void cvt(const void* x, int tx, void* y, int ty, int64_t n, double a_host = 1.0, const double* a_dev = nullptr,
           bool square_dev = false) {
    ew(EW_CVT, x, tx, n * dsize(tx), nullptr, 0, y, ty, n * dsize(ty), n, a_host, a_dev, 0.0, nullptr, square_dev ? 1 : 0);
  }
  void to32plain(const double* x, float* y, int64_t n) { cvt(x, DT_F64, y, DT_F32, n); }
  void scale32(const float* x, float* y, int64_t n, double a_host, const double* a_dev) { cvt(x, DT_F32, y, DT_F32, n, a_host, a_dev); }
  void to64(const float* x, double* y, int64_t n) { cvt(x, DT_F32, y, DT_F64, n); }
  void axpby(const double* x, const double* y, double* z, int64_t n, double a, const double* a_dev,
             double b, const double* b_dev) {
    ew(EW_AXPBY64, x, DT_F64, n * 8, y, n * 8, z, DT_F64, n * 8, n, a, a_dev, b, b_dev);
  }
  // dst[i, j] (ld ldd) = src[i, j] (ld lds), rows x cols, with conversion
  void copy2d(const void* src, int ts, int64_t lds, void* dst, int td, int64_t ldd, int rows, int cols) {
    ew(EW_CVT_2D, src, ts, ((size_t)(rows - 1) * lds + cols) * dsize(ts), nullptr, 0, dst, td,
       ((size_t)(rows - 1) * ldd + cols) * dsize(td), (int64_t)rows * cols, 1.0, nullptr, 0.0, nullptr, lds, ldd, rows, cols);
  }
  void transpose_into(const double* src, int n, double* dst, int64_t ldd) {
    ew(EW_TRANSPOSE_INTO, src, DT_F64, (size_t)n * n * 8, nullptr, 0, dst, DT_F64, ((size_t)(n - 1) * ldd + n) * 8,
       (int64_t)n * n, 1.0, nullptr, 0.0, nullptr, n, ldd, n, 0);
  }
  void symmetrize_lower(double* A, int n) {
    ew(EW_SYMM_LOWER, nullptr, DT_F64, 0, nullptr, 0, A, DT_F64, (size_t)n * n * 8, (int64_t)n * n, 1.0, nullptr, 0.0,
       nullptr, n, 0, n, 0, true);
  }
  // norm_out[0] = sqrt(max(sq[0], 0)); alpha_out[0] = hyper[3] != 0 ? hyper[3] / norm : 1
  void norm_finish(const double* sq, const double* hyper, double* norm_out, double* alpha_out) {
    if (err) return;
    Rec rec{};
    rec.op.kind = OP_EW; rec.op.ew = EW_NORM_FINISH; rec.op.units = 1;
    EwPart& e = rec.op.e;
    e.x = sq; e.y = alpha_out; e.z = norm_out; e.d0 = hyper; e.count = 1;
    rec.rd[rec.nrd++] = range(sq, 8);
    rec.rd[rec.nrd++] = range(hyper, 32);
    rec.wr[rec.nwr++] = range(norm_out, 8);
    rec.wr[rec.nwr++] = range(alpha_out, 8);
    push(rec);
  }
  void adam_finish(const double* sq, double* hyper, double* adam, double* norm_out, double* alpha_out) {
    if (err) return;
    Rec rec{};
    rec.op.kind = OP_EW; rec.op.ew = EW_ADAM_FINISH; rec.op.units = 1;
    EwPart& e = rec.op.e;
    e.x = sq; e.y = alpha_out; e.z = norm_out; e.d0 = hyper; e.d1 = adam; e.count = 1;
    rec.rd[rec.nrd++] = range(sq, 8);
    rec.rd[rec.nrd++] = range(adam, 64);
    rec.wr[rec.nwr++] = range(norm_out, 8);
    rec.wr[rec.nwr++] = range(alpha_out, 8);
    rec.wr[rec.nwr++] = range(hyper + 2, 8);     // the momentum coefficient
    rec.wr[rec.nwr++] = range(adam, 64);         // the state, updated in place
    push(rec);
  }
  void zero64(double* z, int64_t n) { ew(EW_ZERO64, nullptr, DT_F64, 0, nullptr, 0, z, DT_F64, n * 8, n, 0.0, nullptr, 0.0, nullptr); }

  // out[0] = (accumulate ? out[0] : 0) + scale * sum x[i] y[i]   (deterministic two-stage sum)
  void dot(const void* x, int tx, const void* y, int ty, int64_t n, double scale, double* out, int accumulate) {
    if (err || n <= 0) return;
    const int64_t units64 = (n + kEwChunk - 1) / kEwChunk;
    if (units64 > L.dot_slots) {       // the partial count is fixed by kEwChunk: never widen the chunk to make it fit
      rt::set_error("small stage: a dot over %lld elements needs %lld partial slots, the workspace has %d",
                    (long long)n, (long long)units64, L.dot_slots);
      err = 2; return;
    }
    const int units = (int)units64;
    if (dot_off + units > L.dot_slots) { flush(); }
    double* part = p(L.dot_partial) + dot_off;
    dot_off += units;
    Rec rec{};
    rec.op.kind = OP_DOT;
    EwPart& e = rec.op.e;
    e.x = x; e.y = y; e.z = part; e.tx = tx; e.tz = ty; e.count = n;
    rec.op.units = units;
    rec.rd[rec.nrd++] = range(x, n * dsize(tx));
    rec.rd[rec.nrd++] = range(y, n * dsize(ty));
    rec.wr[rec.nwr++] = range(part, (size_t)units * 8);
    push(rec);
    Rec fin{};
    fin.op.kind = OP_DOTFIN;
    EwPart& f = fin.op.e;
    f.x = part; f.z = out; f.count = units; f.s0 = scale; f.p0 = accumulate;
    fin.op.units = 1;
    fin.rd[fin.nrd++] = range(part, (size_t)units * 8);
    if (accumulate) fin.rd[fin.nrd++] = range(out, 8);
    fin.wr[fin.nwr++] = range(out, 8);
    push(fin);
  }

  int spd(const SpdBatch& b, int count, int nmax) {
    flush();
    if (err) return 1;
    size_t smem = ((size_t)nmax * (nmax + 1) / 2 + (size_t)SPD_NB * nmax) * sizeof(double);
    const size_t smem_limit = 227 * 1024 - 3072;      // the kernel also has ~2.7 KB of static shared memory
    if (smem > smem_limit || nmax > 256) {
      rt::set_error("small stage: rank %d exceeds the in-shared-memory Cholesky limit (230)", nmax); return 2; }
    // tensor-core phases need one more [8][n] block; the largest ranks keep the plain fp64 path
    SpdBatch bb = b;
    bb.dmma = (smem + (size_t)SPD_NB * nmax * sizeof(double) <= smem_limit) ? 1 : 0;
    if (bb.dmma) smem += (size_t)SPD_NB * nmax * sizeof(double);
    if (cudaFuncSetAttribute(spd_blocked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      rt::set_error("small stage: cannot raise shared memory to %zu", smem); return 1; }
    spd_blocked_kernel<<<count, SPD_THREADS, smem, s>>>(bb); ++rt::g_launches;
    return 0;
  }
};

int finish(Ctx& c, const char* what) {
  c.flush();
  if (c.err) { if (c.err == 1) rt::set_error("%s: kernel launch failed", what); return 1; }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { rt::set_error("%s: %s", what, cudaGetErrorString(e)); return 1; }
  return 0;
}

// Contraction of a grouped rank-2r core with W_i = [W_ia | W_ib] (each r_i x r_i, given by strides):
//   out = X x(W0a,W1a,W2a) + B0 x(W0b,W1a,W2a) + B1 x(W0a,W1b,W2a) + B2 x(W0a,W1a,W2b)
// evaluated as   D  = X x0 W0a + B0 x0 W0b ;  E1 = B1 x0 W0a ;  E2 = B2 x0 W0a
//                U1 = D x1 W1a + E1 x1 W1b ;  U2 = E2 x1 W1a ;  out = U1 x2 W2a + U2 x2 W2b.
// Buffers are caller-provided; allowed aliases: E2 == E1 iff B2 == B1; U2 may reuse E1 when
// E2 != E1; out may reuse D.
template <typename T>
void grouped_contract(Ctx& c, const T* X, const T* const B[3], const T* const Wa[3],
                      const T* const Wb[3], const int64_t st_o[3], const int64_t st_i[3],
                      T* D, T* E1, T* E2, T* U1, T* U2, T* out) {
  const int d[3] = {c.r(0), c.r(1), c.r(2)};
  c.mode_prod(0, Wa[0], st_o[0], st_i[0], d[0], d[0], X, d, D, 1.0, 0.0);
  c.mode_prod(0, Wb[0], st_o[0], st_i[0], d[0], d[0], B[0], d, D, 1.0, 1.0);
  c.mode_prod(0, Wa[0], st_o[0], st_i[0], d[0], d[0], B[1], d, E1, 1.0, 0.0);
  if (E2 != E1) c.mode_prod(0, Wa[0], st_o[0], st_i[0], d[0], d[0], B[2], d, E2, 1.0, 0.0);
  c.mode_prod(1, Wa[1], st_o[1], st_i[1], d[1], d[1], D, d, U1, 1.0, 0.0);
  c.mode_prod(1, Wb[1], st_o[1], st_i[1], d[1], d[1], E1, d, U1, 1.0, 1.0);
  c.mode_prod(1, Wa[1], st_o[1], st_i[1], d[1], d[1], E2, d, U2, 1.0, 0.0);
  c.mode_prod(2, Wa[2], st_o[2], st_i[2], d[2], d[2], U1, d, out, 1.0, 0.0);
  c.mode_prod(2, Wb[2], st_o[2], st_i[2], d[2], d[2], U2, d, out, 1.0, 1.0);
}

// Records rt_small_prepare's program (the fp64 core, its unfolding Grams, ||core||^2) and fills the batch of the
// factorisation that follows it.  Returns its largest order.
int prepare_program(Ctx& c, const float* core, int sym, SpdBatch& b) {
  const int d[3] = {c.r(0), c.r(1), c.r(2)};
  double* C64 = c.p(c.L.C64);
  c.to64(core, C64, c.L.c);
  for (int i = 0; i < 3; ++i) c.unfold_gram(i, C64, d, C64, d[i], c.p(c.L.Gm[i]), d[i], 1.0, 0.0);
  if (sym) {
    c.axpby(c.p(c.L.Gm[1]), c.p(c.L.Gm[2]), c.p(c.L.Gm[1]), (int64_t)d[1] * d[1], 1.0, nullptr, 1.0, nullptr);
    c.axpby(c.p(c.L.Gm[1]), nullptr, c.p(c.L.Gm[2]), (int64_t)d[1] * d[1], 1.0, nullptr, 0.0, nullptr);
  }
  int nmax = 0;
  for (int i = 0; i < 3; ++i) {
    b.p[i].G = c.p(c.L.Gm[i]); b.p[i].L = nullptr; b.p[i].Linv = nullptr; b.p[i].Ginv = c.p(c.L.Ainv[i]);
    b.p[i].n = d[i];
    nmax = d[i] > nmax ? d[i] : nmax;
  }
  c.dot(C64, DT_F64, C64, DT_F64, c.L.c, 1.0, c.p(c.L.coresq), 0);
  return nmax;
}

// The projection of rt_small_project in two parts.  The head transports the previous direction: pS (fp32, in T6) and
// KC_i (fp64).  It reads neither the factorisation's Grams nor its inverses, nor hyper, so it can run alongside
// rt_small_prepare's factorisation (rt_small_prepare_project).  The tail scales by beta = hyper[2] and applies the
// inverses: pS_beta = beta pS, K_i = beta KC_i Ainv_i, L_i = -M_i K_i.
void project_head(Ctx& c, const float* core, const float* core_old, const float* dS_old, const double* const M[3],
                  int sym) {
  const int d[3] = {c.r(0), c.r(1), c.r(2)};
  // All O(r^4) contractions of the projection run in fp32 (inputs are the fp32 parameters themselves and
  // the result only needs fp32 accuracy); the r x r solves with (S_(i)S_(i)^T)^-1 stay in fp64.
  const float* Cf = core;
  const float* Co = core_old;
  const float* Xo = dS_old;
  float* Mf[3];
  for (int i = 0; i < 3; ++i) Mf[i] = reinterpret_cast<float*>(c.p(c.L.tmpM[i]));
  for (int i = 0; i < (sym ? 2 : 3); ++i) c.to32plain(M[i], Mf[i], 2 * (int64_t)d[i] * d[i]);
  if (sym) Mf[2] = Mf[1];
  const float* Wa[3]; const float* Wb[3]; int64_t st_o[3], st_i[3];
  for (int i = 0; i < 3; ++i) { Wa[i] = Mf[i]; Wb[i] = Mf[i] + d[i]; st_o[i] = 2 * d[i]; st_i[i] = 1; }
  const float* Cb[3] = {Co, Co, Co};
  float* D = c.Tf(2); float* Ta = c.Tf(3); float* U1 = c.Tf(4); float* U2 = c.Tf(5);
  float* pS = c.Tf(6);
  grouped_contract<float>(c, Xo, Cb, Wa, Wb, st_o, st_i, D, Ta, Ta, U1, U2, pS);
  // KC_i (2 r_i x r_i) in fp32 scratch (the eigenvector slots are idle here), converted to fp64 afterwards
  float* KCf[3] = {reinterpret_cast<float*>(c.p(c.L.Vf[0])), reinterpret_cast<float*>(c.p(c.L.Vf[1])),
                   reinterpret_cast<float*>(c.p(c.L.Vf[2]))};
  double* KC[3] = {c.p(c.L.KC[0]), c.p(c.L.KC[1]), c.p(c.L.KC[2])};
  // KC_2 = [U1_(2) ; U2_(2)] C_(2)^T
  c.unfold_gram<float>(2, U1, d, Cf, d[2], KCf[2], d[2], 1.0, 0.0);
  c.unfold_gram<float>(2, U2, d, Cf, d[2], KCf[2] + (int64_t)d[2] * d[2], d[2], 1.0, 0.0);
  // KC_1: V1 = D x2 W2a + Ta x2 W2b ; V2 = Ta x2 W2a     (reuse U1/U2 storage after KC_2)
  // Every intermediate has its own buffer (T0, T1, T7 and both halves are idle during the projection): the levels come
  // from byte-range hazards, so REUSING U1 / U2 / Ta / D here serialised the three KC chains behind each other
  // (16 levels); with private buffers the KC_0 chain starts at level 0 and KC_1 right after the first mode products.
  float* V1 = c.Tf(0); float* V2 = c.Tf(0) + c.L.c;
  c.mode_prod<float>(2, Wa[2], st_o[2], st_i[2], d[2], d[2], D, d, V1, 1.0, 0.0);
  c.mode_prod<float>(2, Wb[2], st_o[2], st_i[2], d[2], d[2], Ta, d, V1, 1.0, 1.0);
  c.mode_prod<float>(2, Wa[2], st_o[2], st_i[2], d[2], d[2], Ta, d, V2, 1.0, 0.0);
  c.unfold_gram<float>(1, V1, d, Cf, d[1], KCf[1], d[1], 1.0, 0.0);
  c.unfold_gram<float>(1, V2, d, Cf, d[1], KCf[1] + (int64_t)d[1] * d[1], d[1], 1.0, 0.0);
  // KC_0: Ea = Co x1 W1a, Eb = Co x1 W1b, F = Xo x1 W1a + Eb ; Z1 = F x2 W2a + Ea x2 W2b ; Z2 = Ea x2 W2a
  float* Ea = c.Tf(1); float* F = c.Tf(1) + c.L.c;
  c.mode_prod<float>(1, Wa[1], st_o[1], st_i[1], d[1], d[1], Co, d, Ea, 1.0, 0.0);
  c.mode_prod<float>(1, Wa[1], st_o[1], st_i[1], d[1], d[1], Xo, d, F, 1.0, 0.0);
  c.mode_prod<float>(1, Wb[1], st_o[1], st_i[1], d[1], d[1], Co, d, F, 1.0, 1.0);
  float* Z1 = c.Tf(7); float* Z2 = c.Tf(7) + c.L.c;
  c.mode_prod<float>(2, Wa[2], st_o[2], st_i[2], d[2], d[2], F, d, Z1, 1.0, 0.0);
  c.mode_prod<float>(2, Wb[2], st_o[2], st_i[2], d[2], d[2], Ea, d, Z1, 1.0, 1.0);
  c.mode_prod<float>(2, Wa[2], st_o[2], st_i[2], d[2], d[2], Ea, d, Z2, 1.0, 0.0);
  c.unfold_gram<float>(0, Z1, d, Cf, d[0], KCf[0], d[0], 1.0, 0.0);
  c.unfold_gram<float>(0, Z2, d, Cf, d[0], KCf[0] + (int64_t)d[0] * d[0], d[0], 1.0, 0.0);
  for (int i = 0; i < 3; ++i) c.to64(KCf[i], KC[i], 2 * (int64_t)d[i] * d[i]);
  if (sym) c.axpby(KC[1], KC[2], KC[1], 2 * (int64_t)d[1] * d[1], 1.0, nullptr, 1.0, nullptr);
}

void project_tail(Ctx& c, const double* const M[3], const double* hyper, int sym, float* pS_beta, double* const K[3],
                  double* const L[3]) {
  const int d[3] = {c.r(0), c.r(1), c.r(2)};
  c.scale32(c.Tf(6), pS_beta, c.L.c, 1.0, hyper + 2);
  const int nm = sym ? 2 : 3;
  for (int i = 0; i < nm; ++i) {
    // K_i = beta * KC_i Ainv_i ;  L_i = -M_i K_i
    c.matmul(c.p(c.L.KC[i]), d[i], false, c.p(c.L.Ainv[i]), d[i], false, K[i], d[i], 2 * d[i], d[i], d[i], 1.0, 0.0,
             hyper + 2);
    c.matmul(M[i], 2 * d[i], false, K[i], d[i], false, L[i], d[i], d[i], d[i], 2 * d[i], -1.0, 0.0);
  }
  if (sym && K[2] && K[2] != K[1]) {
    c.axpby(K[1], nullptr, K[2], 2 * (int64_t)d[1] * d[1], 1.0, nullptr, 0.0, nullptr);
    c.axpby(L[1], nullptr, L[2], (int64_t)d[1] * d[1], 1.0, nullptr, 0.0, nullptr);
  }
}

}  // namespace

extern "C" size_t rt_small_ws_bytes(int r0, int r1, int r2, int B) {
  if (r0 <= 0 || r1 <= 0 || r2 <= 0) return 0;
  return make_layout(r0, r1, r2, B).total;
}

extern "C" int rt_small_prepare(const float* core, int r0, int r1, int r2, int sym, void* small_ws,
                                void* stream) {
  RT_REQUIRE(small_ws != nullptr && r0 > 0 && r1 > 0 && r2 > 0, "rt_small_prepare: bad arguments");
  RT_REQUIRE(!sym || r1 == r2, "rt_small_prepare: SF-Tucker needs r1 == r2");
  Ctx c{make_layout(r0, r1, r2, 0), (char*)small_ws, (cudaStream_t)stream};
  // layout must not depend on B for the persistent slots: they precede every B-dependent slot
  SpdBatch b{};
  const int nmax = prepare_program(c, core, sym, b);
  int rc = c.spd(b, 3, nmax);
  if (rc) return rc;
  return finish(c, "rt_small_prepare");
}

extern "C" int rt_small_prepare_project(const float* core, const float* core_old, const float* dS_old,
                                        const double* M_R, const double* M_S, const double* M_O, int r0, int r1,
                                        int r2, int sym, void* small_ws, void* stream) {
  RT_REQUIRE(small_ws != nullptr && r0 > 0 && r1 > 0 && r2 > 0, "rt_small_prepare_project: bad arguments");
  RT_REQUIRE(!sym || r1 == r2, "rt_small_prepare_project: SF-Tucker needs r1 == r2");
  Ctx c{make_layout(r0, r1, r2, 0), (char*)small_ws, (cudaStream_t)stream};
  SpdBatch b{};
  const int nmax = prepare_program(c, core, sym, b);
  int rc = c.spd(b, 3, nmax);
  if (rc) return rc;
  // The factorisation occupies one SM per problem and leaves the others idle for ~0.3 ms at r = 200.  The head runs
  // there, as its programmatic dependent on a grid that fits beside it; its results do not depend on the grid size.
  const double* M[3] = {M_R, M_S, sym ? M_S : M_O};
  project_head(c, core, core_old, dS_old, M, sym);
  c.flush(kExecCtasPerSm * std::max(1, rt::sm_count() - 3), Launch::kAfterPrimary);
  return finish(c, "rt_small_prepare_project");
}

extern "C" size_t rt_small_ainv_offset(int mode, int r0, int r1, int r2) {
  if (mode < 0 || mode > 2) return (size_t)-1;
  return make_layout(r0, r1, r2, 0).Ainv[mode];
}

extern "C" int rt_rows_times_ainv(const float* A, int m, int mode, int r0, int r1, int r2, float* C,
                                  void* small_ws, void* stream) {
  RT_REQUIRE(mode >= 0 && mode < 3 && m >= 0, "rt_rows_times_ainv: bad arguments");
  if (m == 0) return 0;
  Layout L = make_layout(r0, r1, r2, 0);
  const int r = L.r[mode];
  const double* K = (const double*)((char*)small_ws + L.Ainv[mode]);
  const size_t smem = (size_t)4 * r * sizeof(float);
  rows_times_mat_kernel<<<cdiv(m, 4), 256, smem, (cudaStream_t)stream>>>(A, m, r, K, C);
  RT_LAUNCH_CHECK();
  return 0;
}

extern "C" int rt_small_grad(const float* core, const float* d_core, const float* qp, const float* H,
                             const float* r_rows, const float* s_rows, const float* dr_rows,
                             const float* ds_rows, const double* bce_sum, double inv_count,
                             const double* hyper, int B, int r0, int r1, int r2, int sym, float* dS_g,
                             double* loss_total, float* drA, float* dsA, double* P_R, double* P_S,
                             double* P_O, void* small_ws, void* stream) {
  RT_REQUIRE(small_ws != nullptr && B > 0, "rt_small_grad: bad arguments");
  Ctx c{make_layout(r0, r1, r2, B), (char*)small_ws, (cudaStream_t)stream};
  // dS_g = d_core + 2 reg core
  c.ew(EW_GRAD_CORE, d_core, DT_F32, c.L.c * 4, core, c.L.c * 4, dS_g, DT_F32, c.L.c * 4, c.L.c, 1.0, hyper, 0.0, nullptr,
       0, 0, 0, 0, false, 32);
  // loss_total = bce_sum * inv_count + reg * ||core||^2
  c.axpby(bce_sum, c.p(c.L.coresq), loss_total, 1, inv_count, nullptr, 1.0, hyper + 1);
  // drA = dr_rows A_R^-1, dsA = ds_rows A_S^-1   (fp32 rows times the fp64 inverses of rt_small_prepare)
  auto rows_ainv = [&](const float* rows, int mode, float* out) {
    const int r = c.r(mode);
    c.gemm_any(rows, DT_F32, c.p(c.L.Ainv[mode]), DT_F64, out, DT_F32, B, r, 1, r, r, 0, 1, 0, r, 1, r, 1, 1, 0, 0, 0,
               1.0, 0.0);
  };
  rows_ainv(dr_rows, 0, drA);
  rows_ainv(ds_rows, 1, dsA);
  // P_i = -(U_i^T g_i A_i): the Gram of the gathered rows with the A-scaled gradient rows (contraction over the batch)
  auto gram_rows = [&](const float* X, const float* Y, int r, double* out, double alpha, double beta) {
    c.gemm_any(X, DT_F32, Y, DT_F32, out, DT_F64, r, r, 1, B, 1, 0, r, 0, r, 1, r, 1, 1, 0, 0, 0, alpha, beta);
  };
  gram_rows(r_rows, drA, r0, P_R, -1.0, 0.0);
  gram_rows(s_rows, dsA, r1, P_S, -1.0, 0.0);
  if (sym) {
    gram_rows(H, qp, r2, P_S, -1.0, 1.0);
    if (P_O && P_O != P_S) c.axpby(P_S, nullptr, P_O, (int64_t)r1 * r1, 1.0, nullptr, 0.0, nullptr);
  } else {
    gram_rows(H, qp, r2, P_O, -1.0, 0.0);
  }
  return finish(c, "rt_small_grad");
}

// The norm's program.  With `tail` it also records the projection's tail (project_tail) after it: for TuckerAdam
// the tail reads the momentum coefficient that adam_finish writes.
struct ProjectTail { const double* M[3]; float* pS_beta; double* K[3]; double* L[3]; };

static int small_norm_impl(const float* dS_g, const double* gram_R, const double* gram_S, const double* gram_O,
                           double* hyper, double* adam, int r0, int r1, int r2, int sym, double* norm_out,
                           double* alpha_out, const ProjectTail* tail, void* small_ws, void* stream) {
  Ctx c{make_layout(r0, r1, r2, 0), (char*)small_ws, (cudaStream_t)stream};
  double* sq = c.p(c.L.scal);
  c.dot(dS_g, DT_F32, dS_g, DT_F32, c.L.c, 1.0, sq, 0);
  c.dot(gram_R, DT_F64, c.p(c.L.Gm[0]), DT_F64, (int64_t)r0 * r0, 1.0, sq, 1);
  c.dot(gram_S, DT_F64, c.p(c.L.Gm[1]), DT_F64, (int64_t)r1 * r1, 1.0, sq, 1);
  if (!sym) c.dot(gram_O, DT_F64, c.p(c.L.Gm[2]), DT_F64, (int64_t)r2 * r2, 1.0, sq, 1);
  if (adam) c.adam_finish(sq, hyper, adam, norm_out, alpha_out);
  else c.norm_finish(sq, hyper, norm_out, alpha_out);
  if (tail) project_tail(c, tail->M, hyper, sym, tail->pS_beta, tail->K, tail->L);
  return finish(c, tail ? "rt_small_norm_project" : "rt_small_norm");
}

extern "C" int rt_small_norm(const float* dS_g, const double* gram_R, const double* gram_S,
                             const double* gram_O, const double* hyper, int r0, int r1, int r2, int sym,
                             double* norm_out, double* alpha_out, void* small_ws, void* stream) {
  RT_REQUIRE(small_ws != nullptr, "rt_small_norm: workspace is NULL");
  return small_norm_impl(dS_g, gram_R, gram_S, gram_O, const_cast<double*>(hyper), nullptr, r0, r1, r2, sym, norm_out,
                         alpha_out, nullptr, small_ws, stream);
}

extern "C" int rt_small_norm_adam(const float* dS_g, const double* gram_R, const double* gram_S,
                                  const double* gram_O, double* hyper, double* adam, int r0, int r1, int r2, int sym,
                                  double* norm_out, double* alpha_out, void* small_ws, void* stream) {
  RT_REQUIRE(small_ws != nullptr && adam != nullptr, "rt_small_norm_adam: NULL argument");
  return small_norm_impl(dS_g, gram_R, gram_S, gram_O, hyper, adam, r0, r1, r2, sym, norm_out, alpha_out, nullptr,
                         small_ws, stream);
}

extern "C" int rt_small_norm_project(const float* dS_g, const double* gram_R, const double* gram_S,
                                     const double* gram_O, double* hyper, double* adam, const double* M_R,
                                     const double* M_S, const double* M_O, int r0, int r1, int r2, int sym,
                                     double* norm_out, double* alpha_out, float* pS_beta, double* K_R, double* K_S,
                                     double* K_O, double* L_R, double* L_S, double* L_O, void* small_ws,
                                     void* stream) {
  RT_REQUIRE(small_ws != nullptr, "rt_small_norm_project: workspace is NULL");
  const ProjectTail tail{{M_R, M_S, sym ? M_S : M_O}, pS_beta, {K_R, K_S, K_O}, {L_R, L_S, L_O}};
  return small_norm_impl(dS_g, gram_R, gram_S, gram_O, hyper, adam, r0, r1, r2, sym, norm_out, alpha_out, &tail,
                         small_ws, stream);
}

extern "C" int rt_small_project(const float* core, const float* core_old, const float* dS_old,
                                const double* M_R, const double* M_S, const double* M_O,
                                const double* hyper, int r0, int r1, int r2, int sym, float* pS_beta,
                                double* K_R, double* K_S, double* K_O, double* L_R, double* L_S,
                                double* L_O, void* small_ws, void* stream) {
  RT_REQUIRE(small_ws != nullptr, "rt_small_project: workspace is NULL");
  Ctx c{make_layout(r0, r1, r2, 0), (char*)small_ws, (cudaStream_t)stream};
  const double* M[3] = {M_R, M_S, sym ? M_S : M_O};
  double* const K[3] = {K_R, K_S, K_O};
  double* const L[3] = {L_R, L_S, L_O};
  project_head(c, core, core_old, dS_old, M, sym);
  project_tail(c, M, hyper, sym, pS_beta, K, L);
  return finish(c, "rt_small_project");
}

extern "C" int rt_small_retract(const float* core, const float* dS_dir, const double* gram_R,
                                const double* gram_S, const double* gram_O, const double* hyper, int r0,
                                int r1, int r2, int sym, float* core_new, double* Z1_R, double* Z2_R,
                                double* Z1_S, double* Z2_S, double* Z1_O, double* Z2_O, double* Mn_R,
                                double* Mn_S, double* Mn_O, void* small_ws, void* stream) {
  RT_REQUIRE(small_ws != nullptr, "rt_small_retract: workspace is NULL");
  Ctx c{make_layout(r0, r1, r2, 0), (char*)small_ws, (cudaStream_t)stream};
  cudaStream_t s = c.s;
  const int d[3] = {r0, r1, r2};
  const double* gram[3] = {gram_R, gram_S, sym ? gram_S : gram_O};
  double* Z1[3] = {Z1_R, Z1_S, Z1_O};
  double* Z2[3] = {Z2_R, Z2_S, Z2_O};
  const double* lr = hyper + 0;
  double* C = c.p(c.L.C64);
  // C' = core - lr dS_dir
  double* Cp = c.T(0);
  c.ew(EW_CORE_MINUS_LR, core, DT_F32, c.L.c * 4, dS_dir, c.L.c * 4, Cp, DT_F64, c.L.c * 8, c.L.c, 1.0, lr, 0.0, nullptr);
  // Gamma_i = lr^2 Gram_i = L_i L_i^T ; R_i = L_i^T
  SpdBatch b{};
  int nmax = 0;
  const int nm = sym ? 2 : 3;
  for (int i = 0; i < nm; ++i) {
    const int n2 = d[i] * d[i];
    c.cvt(gram[i], DT_F64, c.p(c.L.Gs[i]), DT_F64, n2, 1.0, lr, true);
    b.p[i].G = c.p(c.L.Gs[i]); b.p[i].L = c.p(c.L.GL[i]); b.p[i].Linv = c.p(c.L.GLinv[i]);
    b.p[i].Ginv = nullptr; b.p[i].n = d[i];
    nmax = d[i] > nmax ? d[i] : nmax;
  }
  int rc = c.spd(b, nm, nmax);
  if (rc) return rc;
  const double* Lc[3] = {c.p(c.L.GL[0]), c.p(c.L.GL[1]), c.p(c.L.GL[sym ? 1 : 2])};
  const double* Linv[3] = {c.p(c.L.GLinv[0]), c.p(c.L.GLinv[1]), c.p(c.L.GLinv[sym ? 1 : 2])};
  // B_i = C x_i R_i,  R_i = L_i^T  => M[o,i] = L[i,o]: strides (sm_o, sm_i) = (1, d)
  double* Bk[3] = {c.T(1), c.T(2), c.T(3)};
  for (int i = 0; i < 3; ++i) c.mode_prod(i, Lc[i], 1, d[i], d[i], d[i], C, d, Bk[i], 1.0, 0.0);
  // unfolding Grams N_i (2r_i x 2r_i)
  double* Nn[3] = {c.p(c.L.Nn[0]), c.p(c.L.Nn[1]), c.p(c.L.Nn[2])};
  for (int i = 0; i < 3; ++i) {
    const int n = 2 * d[i];
    c.zero64(Nn[i], (int64_t)n * n);
    c.unfold_gram(i, Cp, d, Cp, d[i], Nn[i], n, 1.0, 0.0);
    for (int j = 0; j < 3; ++j)
      if (j != i) c.unfold_gram(i, Bk[j], d, Bk[j], d[i], Nn[i], n, 1.0, 1.0);
    c.unfold_gram(i, Bk[i], d, Cp, d[i], Nn[i] + (int64_t)d[i] * n, n, 1.0, 0.0);
    c.unfold_gram(i, Bk[i], d, Bk[i], d[i], Nn[i] + (int64_t)d[i] * n + d[i], n, 1.0, 0.0);
    c.symmetrize_lower(Nn[i], n);
  }
  if (sym) c.axpby(Nn[1], Nn[2], Nn[1], 4 * (int64_t)d[1] * d[1], 1.0, nullptr, 1.0, nullptr);
  c.flush();
  if (c.err) return finish(c, "rt_small_retract");
  const double* Ain[3]; int nn[3]; int rr[3]; int ldy[3]; double* Yv[3]; void* sws[3];
  for (int i = 0; i < nm; ++i) {
    Ain[i] = Nn[i]; nn[i] = 2 * d[i]; rr[i] = d[i]; ldy[i] = 2 * d[i]; Yv[i] = c.p(c.L.Vf[i]);
    sws[i] = c.base + c.L.sub[i];
  }
  if ((rc = rt::subspace_batch(nm, Ain, nn, rr, Yv, ldy, sws, c.base + c.L.sub_shared, nullptr, s))) return rc;
  // Y_i = V_i[:, :r_i]  (2r_i x r_i, row stride 2r_i);  W_i = Y_i^T = [Y_ia^T | Y_ib^T]
  const double* Y[3] = {c.p(c.L.Vf[0]), c.p(c.L.Vf[1]), c.p(c.L.Vf[sym ? 1 : 2])};
  // core_new = T x_i Y_i^T through the block structure, in fp32 (the output is fp32): fp32 images of C', B_k
  // and of Y_i (dense [2 r_i, r_i]) live in the scratch temporaries T4..T7 (8 x c floats) and tmpM.
  float* CpF = c.Tf(4); float* BkF[3] = {c.Tf(4) + c.L.c, c.Tf(5), c.Tf(5) + c.L.c};
  c.to32plain(Cp, CpF, c.L.c);
  for (int i = 0; i < 3; ++i) c.to32plain(Bk[i], BkF[i], c.L.c);
  float* Yf[3];
  for (int i = 0; i < 3; ++i) Yf[i] = reinterpret_cast<float*>(c.p(c.L.tmpM[i]));
  for (int i = 0; i < nm; ++i) {
    c.copy2d(Y[i], DT_F64, 2 * d[i], Yf[i], DT_F32, d[i], 2 * d[i], d[i]);
  }
  if (sym) Yf[2] = Yf[1];
  const float* Wa[3]; const float* Wb[3]; int64_t st_o[3], st_i[3];
  for (int i = 0; i < 3; ++i) {
    Wa[i] = Yf[i];                              // W_ia[o, k] = Y[k, o]      -> strides (1, r_i)
    Wb[i] = Yf[i] + (int64_t)d[i] * d[i];       // W_ib[o, k] = Y[r_i + k, o]
    st_o[i] = 1; st_i[i] = d[i];
  }
  const float* Cb[3] = {BkF[0], BkF[1], BkF[2]};
  float* Dn = c.Tf(6); float* E1 = c.Tf(6) + c.L.c; float* E2 = c.Tf(7); float* U1n = c.Tf(7) + c.L.c;
  // U2 reuses E1 (dead once U1 exists), the result reuses D
  grouped_contract<float>(c, CpF, Cb, Wa, Wb, st_o, st_i, Dn, E1, E2, U1n, E1, Dn);
  c.cvt(Dn, DT_F32, core_new, DT_F32, c.L.c);
  // Z1_i = Y_ia ; Z2_i = -lr * L_i^-T Y_ib
  for (int i = 0; i < nm; ++i) {
    const int64_t n = 2 * d[i];
    c.matmul(Linv[i], d[i], true, Y[i] + (int64_t)d[i] * n, n, false, Z2[i], d[i], d[i], d[i], d[i], -1.0, 0.0, lr);
    c.copy2d(Y[i], DT_F64, n, Z1[i], DT_F64, d[i], d[i], d[i]);
  }
  // Transport Grams of the NEXT fit() without touching N-sized data (SURVEY App. A.6): with U^T U = I and
  // U^T dV = 0,  U_new^T [U | dV] = [Z1^T | Z2^T (dV^T dV)]   (r_i x 2 r_i)
  double* Mn[3] = {Mn_R, Mn_S, Mn_O};
  for (int i = 0; i < nm; ++i) {
    if (!Mn[i]) continue;
    const int64_t n2 = 2 * d[i];
    c.transpose_into(Z1[i], d[i], Mn[i], n2);
    c.matmul(Z2[i], d[i], true, gram[i], d[i], false, Mn[i] + d[i], n2, d[i], d[i], d[i], 1.0, 0.0);
  }
  if (sym && Z1_O && Z1_O != Z1_S) {
    c.axpby(Z1_S, nullptr, Z1_O, (int64_t)d[1] * d[1], 1.0, nullptr, 0.0, nullptr);
    c.axpby(Z2_S, nullptr, Z2_O, (int64_t)d[1] * d[1], 1.0, nullptr, 0.0, nullptr);
  }
  // SF-Tucker: a separate Mn_O receives the shared mode's transport Gram, as Z1_O / Z2_O do
  if (sym && Mn_S && Mn_O && Mn_O != Mn_S) c.axpby(Mn_S, nullptr, Mn_O, 2 * (int64_t)d[1] * d[1], 1.0, nullptr, 0.0, nullptr);
  return finish(c, "rt_small_retract");
}
