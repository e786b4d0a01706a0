// C-ABI entry points that build tap-GEMM descriptors (see include/fishdiff_b200.h for the contract).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstring>
#include "fd_common.cuh"
#include "fd_host.h"

namespace {
thread_local char g_err[1024] = "";
std::atomic<long long> g_launches{0};

void set_prec(FdTapGemm& p, int prec) { p.prec = prec & 0xF; p.single = (prec & FD_SINGLE) ? 1 : 0; }
void init_desc(FdTapGemm& p) { memset(&p, 0, sizeof(p)); p.acc_scale = 1.f; p.post_scale = 1.f; p.planes_scale = 1.f; p.res_scale = 1.f; }

void set_src(FdTapGemm& p, int i, const uint16_t* ptr, int C) {
  p.src[i] = ptr;
  p.src_C[i] = C;
  p.src_rs[i] = C;
  p.src_bs[i] = (long long)p.T * C;
  p.src_ps[i] = (long long)p.B * p.T * C;
}

// ---- optional per-launch device timing (bench.py roofline): event pairs around every tap-GEMM launch
constexpr int PROF_MAX = 1 << 16;
bool g_prof_on = false;
int g_prof_n = 0;
cudaEvent_t* g_prof_ev = nullptr;   // 2 * PROF_MAX events, created lazily
int g_prof_kind[PROF_MAX];

}  // namespace

void fd_prof_begin(int kind, cudaStream_t st) {
  if (!g_prof_on || g_prof_n >= PROF_MAX) return;
  if (g_prof_ev == nullptr) {
    g_prof_ev = new cudaEvent_t[2 * PROF_MAX];
    for (int i = 0; i < 2 * PROF_MAX; ++i) g_prof_ev[i] = nullptr;
  }
  if (g_prof_ev[2 * g_prof_n] == nullptr) {
    cudaEventCreate(&g_prof_ev[2 * g_prof_n]);
    cudaEventCreate(&g_prof_ev[2 * g_prof_n + 1]);
  }
  g_prof_kind[g_prof_n] = kind;
  cudaEventRecord(g_prof_ev[2 * g_prof_n], st);
}
void fd_prof_end(cudaStream_t st) {
  if (!g_prof_on || g_prof_n >= PROF_MAX) return;
  cudaEventRecord(g_prof_ev[2 * g_prof_n + 1], st);
  ++g_prof_n;
}

namespace {

int run(const FdTapGemm& p, int backend, cudaStream_t st) {
  int rc;
  fd_prof_begin(p.epi * 2 + (backend == FD_BACKEND_TC ? 0 : 1), st);
  if (backend == FD_BACKEND_TC) {
    rc = fd_tapgemm_tc_launch(p, st);
  } else if (backend == FD_BACKEND_SIMT) {
    rc = fd_tapgemm_simt_launch(p, st);
  } else {
    fd_set_error("unknown backend %d", backend);
    return -2;
  }
  fd_prof_end(st);
  if (rc == 0) fd_count_launch(1);
  return rc;
}
}  // namespace

void fd_count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

namespace { thread_local int g_target_dev = -1; int g_sms[FD_MAX_DEVICES] = {0}; }

FdDeviceGuard::FdDeviceGuard() {
  if (g_target_dev < 0) return;
  if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; return; }
  if (prev != g_target_dev && cudaSetDevice(g_target_dev) == cudaSuccess) switched = true;
}
FdDeviceGuard::~FdDeviceGuard() {
  if (switched) cudaSetDevice(prev);
}
int fd_current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= FD_MAX_DEVICES) dev = 0;
  return dev;
}
int fd_device_sms(int dev) {
  if (g_sms[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    g_sms[dev] = n;
  }
  return g_sms[dev];
}

extern "C" {

void fd_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

const char* fd_last_error(void) { return g_err; }
void fd_set_device(int device) { g_target_dev = (device >= 0 && device < FD_MAX_DEVICES) ? device : -1; }
int fd_abi_version(void) { return FD_ABI_VERSION; }
long long fd_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

void fd_prof_enable(int on) {
  g_prof_on = on != 0;
  g_prof_n = 0;
}

int fd_prof_collect(double* ms_sum, long long* count, int nkinds) {
  FD_CHECK_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < nkinds; ++k) { ms_sum[k] = 0.0; count[k] = 0; }
  for (int i = 0; i < g_prof_n; ++i) {
    float ms = 0.f;
    FD_CHECK_CUDA(cudaEventElapsedTime(&ms, g_prof_ev[2 * i], g_prof_ev[2 * i + 1]));
    const int k = g_prof_kind[i];
    if (k < nkinds) { ms_sum[k] += ms; count[k] += 1; }
  }
  const int n = g_prof_n;
  g_prof_n = 0;
  return n >= PROF_MAX ? 1 : 0;
}

int fd_tc_supported_linear(int n_total, int k_seg, int num_seg) {
  FdTapGemm p;
  init_desc(p);
  p.B = 1; p.T = 128; p.n_total = n_total; p.num_seg = num_seg; p.k_total = k_seg * num_seg;
  p.epi = FD_EPI_LINEAR;
  if (num_seg < 1 || num_seg > FD_MAX_SEG) return 0;
  for (int s = 0; s < num_seg; ++s) { p.seg[s].src = 0; p.seg[s].k_len = k_seg; }
  set_src(p, 0, reinterpret_cast<const uint16_t*>(16), k_seg);
  return fd_tapgemm_tc_supported(p);
}

static int wavenet_block(const uint16_t* x_planes, uint16_t* x_out_planes, const uint16_t* cond_planes,
                         const float* cond_term, uint16_t* z_planes, uint16_t* y_planes, const uint16_t* w1, const uint16_t* w2,
                         const float* gb_full, const float* gb_lo, const float* gb_hi, int gb_bstride, const float* b2,
                         float* skip_f32, uint16_t* skip_planes, float skip_scale, int B, int T, int C, int E,
                         int dilation, int gate_tile, float w1_inv_scale, float w2_inv_scale, int flags, int prec,
                         int backend, void* stream);

int fd_wavenet_block_fwd(uint16_t* x_planes, const uint16_t* cond_planes, uint16_t* z_planes, const uint16_t* w1,
                         const uint16_t* w2, const float* gb_full, const float* gb_lo, const float* gb_hi,
                         int gb_bstride, const float* b2, float* skip_f32, uint16_t* skip_planes, float skip_scale,
                         int B, int T, int C, int E, int dilation, int gate_tile, float w1_inv_scale,
                         float w2_inv_scale, int flags, int prec, int backend, void* stream) {
  FD_DEVICE_GUARD();
  return wavenet_block(x_planes, nullptr, cond_planes, nullptr, z_planes, nullptr, w1, w2, gb_full, gb_lo, gb_hi, gb_bstride, b2,
                       skip_f32, skip_planes, skip_scale, B, T, C, E, dilation, gate_tile, w1_inv_scale, w2_inv_scale,
                       flags, prec, backend, stream);
}

int fd_wavenet_block_fwd_train(const uint16_t* x_planes, uint16_t* x_out_planes, const uint16_t* cond_planes,
                               uint16_t* z_planes, uint16_t* y_planes, const uint16_t* w1, const uint16_t* w2,
                               const float* gb_full, const float* gb_lo, const float* gb_hi, int gb_bstride,
                               const float* b2, float* skip_f32, uint16_t* skip_planes, float skip_scale, int B, int T,
                               int C, int E, int dilation, int gate_tile, float w1_inv_scale, float w2_inv_scale,
                               int flags, int prec, int backend, void* stream) {
  FD_DEVICE_GUARD();
  FD_REQUIRE(x_out_planes != nullptr && y_planes != nullptr, "fd_wavenet_block_fwd_train: x_out / y planes required");
  return wavenet_block(x_planes, x_out_planes, cond_planes, nullptr, z_planes, y_planes, w1, w2, gb_full, gb_lo, gb_hi,
                       gb_bstride, b2, skip_f32, skip_planes, skip_scale, B, T, C, E, dilation, gate_tile, w1_inv_scale,
                       w2_inv_scale, flags, prec, backend, stream);
}

static int wavenet_block(const uint16_t* x_planes, uint16_t* x_out_planes, const uint16_t* cond_planes,
                         const float* cond_term, uint16_t* z_planes, uint16_t* y_planes, const uint16_t* w1, const uint16_t* w2,
                         const float* gb_full, const float* gb_lo, const float* gb_hi, int gb_bstride, const float* b2,
                         float* skip_f32, uint16_t* skip_planes, float skip_scale, int B, int T, int C, int E,
                         int dilation, int gate_tile, float w1_inv_scale, float w2_inv_scale, int flags, int prec,
                         int backend, void* stream) {
  FD_REQUIRE(B > 0 && T > 0 && C > 0 && E > 0 && dilation > 0, "fd_wavenet_block_fwd: bad shape");
  FD_REQUIRE(C % 8 == 0 && E % 8 == 0, "fd_wavenet_block_fwd: C=%d, E=%d must be multiples of 8", C, E);
  cudaStream_t st = (cudaStream_t)stream;
  // ---- GEMM1: dilated conv (3 taps) + conditioner projection + gate.  With cond_term (W_cond . cond computed once per
  //      sampler call, fd_wavenet_cond_term) the launch reads only the tap columns [0, 3C) of the packed W1 and adds the
  //      conditioner term in the epilogue.
  FdTapGemm p;
  init_desc(p);
  p.B = B; p.T = T; set_prec(p, prec);
  p.n_total = 2 * C; p.k_total = 3 * C + E; p.num_seg = cond_term != nullptr ? 3 : 4;
  p.seg[0] = FdSeg{0, -dilation, 0, C};
  p.seg[1] = FdSeg{0, 0, 0, C};
  p.seg[2] = FdSeg{0, dilation, 0, C};
  p.seg[3] = FdSeg{1, 0, 0, E};
  set_src(p, 0, x_planes, C);
  if (cond_term != nullptr) p.addend = cond_term;
  else set_src(p, 1, cond_planes, E);
  p.w = w1; p.acc_scale = w1_inv_scale;
  p.epi = FD_EPI_GATE;
  p.gbias_full = gb_full; p.gbias_lo = gb_lo; p.gbias_hi = gb_hi; p.gbias_bstride = gb_bstride;
  p.dil = dilation; p.gate_tile = gate_tile; p.C = C;
  p.out_planes = z_planes;
  p.y_planes = y_planes;
  int rc = run(p, backend, st);
  if (rc) return rc;
  // ---- GEMM2: output projection + residual / skip
  FdTapGemm q;
  init_desc(q);
  q.B = B; q.T = T; set_prec(q, prec);
  q.n_total = 2 * C; q.k_total = C; q.num_seg = 1;
  q.seg[0] = FdSeg{0, 0, 0, C};
  set_src(q, 0, z_planes, C);
  q.w = w2; q.acc_scale = w2_inv_scale;
  q.epi = FD_EPI_RES_SKIP;
  q.bias = b2; q.bias_bstride = 0;
  q.x_planes = const_cast<uint16_t*>(x_planes); q.x_out_planes = x_out_planes; q.skip_f32 = skip_f32; q.skip_planes = skip_planes; q.skip_scale = skip_scale;
  q.first_layer = flags & 1; q.last_layer = (flags >> 1) & 1; q.C = C;
  return run(q, backend, st);
}

int fd_wavenet_fwd(const fd_wavenet_fwd_desc* d, void* stream) {
  FD_DEVICE_GUARD();
  FD_REQUIRE(d != nullptr, "fd_wavenet_fwd: null descriptor");
  FD_REQUIRE(d->L >= 1 && d->L <= 64, "fd_wavenet_fwd: L=%d out of range (1..64)", d->L);
  FD_REQUIRE(d->Bs == 1 || d->Bs == d->B, "fd_wavenet_fwd: Bs=%d must be 1 or B=%d", d->Bs, d->B);
  const int B = d->B, T = d->T, M = d->M, C = d->C, E = d->E, L = d->L, Bs = d->Bs;
  int rc = fd_wavenet_step_mlp(d->steps, d->mlp_w0, d->mlp_b0, d->mlp_w1, d->mlp_b1, d->s, d->mlp_ws, Bs, C, stream);
  if (rc) return rc;
  float* gb_full = d->gb;
  float* gb_lo = d->gb + (size_t)L * Bs * 2 * C;
  float* gb_hi = d->gb + (size_t)2 * L * Bs * 2 * C;
  rc = fd_wavenet_gate_bias(d->s, d->wd, d->bd, d->w1p_f32, d->bias_sum, gb_full, gb_lo, gb_hi, d->gb_ws, L, Bs, C,
                            3 * C + E, stream);
  if (rc) return rc;
  fd_conv_desc cd;
  memset(&cd, 0, sizeof(cd));
  cd.B = B; cd.T = T; cd.ntaps = 1; cd.shifts[0] = 0;
  cd.post_scale = 1.f; cd.planes_scale = 1.f; cd.prec = d->prec; cd.backend = d->backend;
  // head: relu(input_projection(x)), masked rows zeroed (wavenet.py:211-218)
  cd.in_planes = d->x_planes; cd.w_planes = d->w_in; cd.bias = d->b_in; cd.row_mask = d->x_mask;
  cd.out_planes = d->xr; cd.Cin = M; cd.N = C; cd.w_inv_scale = d->w_in_inv; cd.act = 1;
  rc = fd_conv_cl_fwd(&cd, stream);
  if (rc) return rc;
  const int gb_stride = Bs > 1 ? 2 * C : 0;
  const float skip_scale = 1.f / sqrtf((float)L);
  for (int l = 0; l < L; ++l) {
    const int flags = (l == 0 ? 1 : 0) | (l == L - 1 ? 2 : 0);
    const size_t go = (size_t)l * Bs * 2 * C;
    const float* ct = d->cond_term != nullptr ? d->cond_term + (size_t)l * B * T * 2 * C : nullptr;
    rc = wavenet_block(d->xr, nullptr, d->cond_planes, ct, d->z, nullptr, d->w1 + (size_t)l * d->w1_lstride,
                       d->w2 + (size_t)l * d->w2_lstride, gb_full + go, gb_lo + go, gb_hi + go, gb_stride,
                       d->b2 + (size_t)l * d->b2_lstride, d->skip_f32, d->skip_planes, skip_scale, B, T, C, E,
                       d->dilation[l], d->gate_tile, d->w1_inv[l], d->w2_inv[l], flags, d->prec, d->backend, stream);
    if (rc) return rc;
  }
  // tail: relu(skip_projection(sum / sqrt(L))) -> output_projection, masked rows zeroed (wavenet.py:228-234)
  cd.in_planes = d->skip_planes; cd.w_planes = d->w_skip; cd.bias = d->b_skip; cd.row_mask = nullptr;
  cd.out_planes = d->z; cd.out_f32 = nullptr; cd.Cin = C; cd.N = C; cd.w_inv_scale = d->w_skip_inv; cd.act = 1;
  rc = fd_conv_cl_fwd(&cd, stream);
  if (rc) return rc;
  cd.in_planes = d->z; cd.w_planes = d->w_out; cd.bias = d->b_out; cd.row_mask = d->x_mask;
  cd.out_planes = nullptr; cd.out_f32 = d->out; cd.Cin = C; cd.N = M; cd.w_inv_scale = d->w_out_inv; cd.act = 0;
  return fd_conv_cl_fwd(&cd, stream);
}

int fd_wavenet_cond_term(const uint16_t* cond_planes, const uint16_t* w1, long long w1_lstride, const float* w1_inv,
                         float* cond_term, int L, int B, int T, int C, int E, int prec, int backend, void* stream) {
  FD_DEVICE_GUARD();
  FD_REQUIRE(L >= 1 && L <= 64, "fd_wavenet_cond_term: L=%d out of range (1..64)", L);
  FD_REQUIRE(B > 0 && T > 0 && C > 0 && E > 0, "fd_wavenet_cond_term: bad shape");
  FD_REQUIRE(C % 8 == 0 && E % 8 == 0, "fd_wavenet_cond_term: C=%d, E=%d must be multiples of 8", C, E);
  for (int l = 0; l < L; ++l) {
    FdTapGemm p;
    init_desc(p);
    p.B = B; p.T = T; set_prec(p, prec);
    p.n_total = 2 * C; p.k_total = 3 * C + E; p.num_seg = 1;
    p.seg[0] = FdSeg{0, 0, 0, E};
    set_src(p, 0, cond_planes, E);
    p.w = w1 + (size_t)l * w1_lstride; p.w_kshift = 3 * C;   // the conditioner columns of the packed W1
    p.acc_scale = w1_inv[l];
    p.epi = FD_EPI_LINEAR;
    p.out_f32 = cond_term + (size_t)l * B * T * 2 * C;
    const int rc = run(p, backend, (cudaStream_t)stream);
    if (rc) return rc;
  }
  return 0;
}

int fd_conv_cl_fwd(const fd_conv_desc* d, void* stream) {
  FD_DEVICE_GUARD();
  FD_REQUIRE(d != nullptr, "fd_conv_cl_fwd: null descriptor");
  FD_REQUIRE(d->ntaps >= 1 && d->ntaps <= FD_MAX_SEG, "fd_conv_cl_fwd: ntaps=%d out of range", d->ntaps);
  FD_REQUIRE(d->B > 0 && d->T > 0 && d->Cin > 0 && d->N > 0, "fd_conv_cl_fwd: bad shape");
  FdTapGemm p;
  init_desc(p);
  p.B = d->B; p.T = d->T; set_prec(p, d->prec);
  p.n_total = d->N; p.k_total = d->ntaps * d->Cin; p.num_seg = d->ntaps;
  for (int j = 0; j < d->ntaps; ++j) p.seg[j] = FdSeg{0, d->shifts[j], 0, d->Cin};
  set_src(p, 0, d->in_planes, d->Cin);
  p.w = d->w_planes; p.acc_scale = d->w_inv_scale;
  p.epi = FD_EPI_LINEAR;
  p.bias = d->bias; p.bias_bstride = 0;
  p.addend = d->addend; p.res_f32 = d->res_f32; p.res_planes = d->res_planes;
  p.post_scale = d->post_scale; p.out_f32 = d->out_f32; p.out_accum = d->out_accum;
  p.out_planes = d->out_planes; p.planes_scale = d->planes_scale; p.act = d->act; p.act_slope = d->act_slope;
  p.row_mask = d->row_mask;
  return run(p, d->backend, (cudaStream_t)stream);
}

int fd_stft_mag_eps_fwd(const uint16_t* padded, const uint16_t* dft_w, uint16_t* mag_planes, int B, long long Np,
                    int n_fft, int hop, int frames, int NB, float w_inv_scale, float mag_scale, float mag_eps, int prec,
                    int backend, void* stream) {
  FD_DEVICE_GUARD();
  FD_REQUIRE(n_fft % 64 == 0 && hop % 8 == 0 && NB % 128 == 0, "fd_stft_mag_fwd: n_fft=%d hop=%d NB=%d unsupported",
             n_fft, hop, NB);
  const long long pitch = (Np + 7) / 8 * 8;
  FD_REQUIRE((long long)(frames - 1) * hop + n_fft <= Np, "fd_stft_mag_fwd: frames exceed the padded signal");
  FdTapGemm p;
  init_desc(p);
  p.B = B; p.T = frames; set_prec(p, prec);
  p.n_total = 2 * NB; p.k_total = n_fft; p.num_seg = 1;
  p.seg[0] = FdSeg{0, 0, 0, n_fft};
  p.src[0] = padded; p.src_C[0] = n_fft;
  p.src_rs[0] = hop; p.src_bs[0] = pitch; p.src_ps[0] = (long long)B * pitch;
  p.w = dft_w; p.acc_scale = w_inv_scale;
  p.epi = FD_EPI_MAG; p.gate_tile = 256; p.C = NB; p.mag_scale = mag_scale; p.mag_eps = mag_eps;
  p.out_planes = mag_planes;
  return run(p, backend, (cudaStream_t)stream);
}

int fd_stft_mag_fwd(const uint16_t* padded, const uint16_t* dft_w, uint16_t* mag_planes, int B, long long Np,
                    int n_fft, int hop, int frames, int NB, float w_inv_scale, float mag_scale, int prec,
                    int backend, void* stream) {
  return fd_stft_mag_eps_fwd(padded, dft_w, mag_planes, B, Np, n_fft, hop, frames, NB, w_inv_scale, mag_scale, 1e-9f, prec,
                             backend, stream);
}

int fd_gemm_cl_fwd(const fd_gemm_desc* d, void* stream) {
  FD_DEVICE_GUARD();
  FD_REQUIRE(d != nullptr, "fd_gemm_cl_fwd: null descriptor");
  FD_REQUIRE(d->num_seg >= 1 && d->num_seg <= FD_MAX_SEG, "fd_gemm_cl_fwd: num_seg=%d out of range", d->num_seg);
  FD_REQUIRE(d->B > 0 && d->T > 0 && d->n_total > 0 && d->k_total > 0, "fd_gemm_cl_fwd: bad shape");
  FdTapGemm p;
  init_desc(p);
  p.B = d->B; p.T = d->T; set_prec(p, d->prec);
  p.n_total = d->n_total; p.k_total = d->k_total; p.num_seg = d->num_seg;
  for (int j = 0; j < d->num_seg; ++j) {
    FD_REQUIRE(d->seg_src[j] == 0 || d->seg_src[j] == 1, "fd_gemm_cl_fwd: segment %d has bad source", j);
    p.seg[j] = FdSeg{d->seg_src[j], d->seg_shift[j], d->seg_coff[j], d->seg_klen[j]};
  }
  for (int i = 0; i < 2; ++i) {
    if (d->src[i] == nullptr) continue;
    set_src(p, i, d->src[i], d->src_C[i]);
    if (d->src_rs[i] != 0) p.src_rs[i] = d->src_rs[i];
    if (d->src_bs[i] != 0) p.src_bs[i] = d->src_bs[i];
    if (d->src_ps[i] != 0) p.src_ps[i] = d->src_ps[i];
  }
  FD_REQUIRE(p.src[0] != nullptr, "fd_gemm_cl_fwd: src[0] is null");
  p.w = d->w; p.acc_scale = d->w_inv_scale; p.w_kshift = d->w_kshift; p.w_bstride_k = d->w_bstride_k;
  p.epi = FD_EPI_LINEAR;
  p.bias = d->bias; p.bias_bstride = d->bias_bstride;
  if (d->gate_y != nullptr) {
    FD_REQUIRE(d->backend == FD_BACKEND_TC, "fd_gemm_cl_fwd: the fused gate backward runs on the tensor-core back end only");
    FD_REQUIRE(d->out_planes != nullptr && d->gate_tile > 0 && d->n_total % 4 == 0 && (d->gate_tile / 2) % 4 == 0,
               "fd_gemm_cl_fwd: gate backward needs out_planes and a gate tile");
  }
  p.addend = d->addend; p.res_f32 = d->res_f32; p.res_planes = d->res_planes; p.res_scale = d->res_scale;
  p.post_scale = d->post_scale; p.out_f32 = d->out_f32; p.out_accum = d->out_accum;
  p.out_planes = d->out_planes; p.planes_scale = d->planes_scale; p.act = d->act; p.act_slope = d->act_slope;
  p.row_mask = d->row_mask;
  if (d->gate_y != nullptr) {
    p.epi = FD_EPI_GATE_BWD;
    p.y_planes = const_cast<uint16_t*>(d->gate_y); p.gate_tile = d->gate_tile; p.dil = d->gate_dil; p.C = d->n_total;
    p.cs = d->gate_cs; p.cs_edge = d->gate_cs_edge; p.cs_scale = d->gate_cs_scale;
  }
  return run(p, d->backend, (cudaStream_t)stream);
}

}  // extern "C"
