// extern "C" surface for the convolution family: validates an rcv_conv_desc and
// maps conv / transposed-conv forward, dgrad and wgrad onto the two engines
// (RcvIgemm, RcvWgrad).  See include/rcv_b200.h for the contract.
#include <stdarg.h>
#include <string.h>

#include "rcv_common.cuh"

static thread_local char g_err[512] = "";

void rcv_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

long long* g_rcv_prof = nullptr;
/* debug hook (not in the public header): device buffer of >= 4096 int64 that CTA 0 of the
 * tensor-core kernels fills with clock64() samples per pipeline phase; NULL switches it off */
extern "C" void rcv_debug_set_prof(void* buf) { g_rcv_prof = reinterpret_cast<long long*>(buf); }

extern "C" int rcv_version(void) { return RCV_ABI_VERSION; }

extern "C" size_t rcv_det_scratch_bytes(int op, int32_t N, int32_t C, int64_t HW) {
  if (N <= 0 || HW <= 0) return 0;
  switch (op) {
    case RCV_DET_CE_FWD: return N <= 65535 ? rcv_ce_fwd_det_bytes(N, HW) : 0;
    case RCV_DET_CE_WEIGHT_SUM: return rcv_ce_weight_sum_det_bytes((int64_t)N * HW);
    case RCV_DET_DICE_FWD: return N <= 65535 && C >= 2 && C <= 8 ? rcv_dice_fwd_det_bytes(N, C, HW) : 0;
    case RCV_DET_L1_SUM: return rcv_l1_sum_det_bytes((int64_t)N * HW);
    default: return 0;
  }
}
extern "C" const char* rcv_last_error(void) { return g_err; }

namespace {

int validate(const rcv_conv_desc* d, const char* who) {
  RCV_REQUIRE(d != nullptr, RCV_ERR_BAD_ARG, "%s: null desc", who);
  RCV_REQUIRE(d->N > 0 && d->Cin > 0 && d->Cout > 0 && d->H > 0 && d->W > 0, RCV_ERR_BAD_ARG,
              "%s: non-positive dimension", who);
  RCV_REQUIRE(d->Cin <= 1024 && d->Cout <= 1024, RCV_ERR_UNSUPPORTED, "%s: channels > 1024", who);
  if (d->transposed) {
    RCV_REQUIRE(d->ksize == 3 && d->stride == 2 && d->pad == 1 && d->dil == 1, RCV_ERR_UNSUPPORTED,
                "%s: transposed conv supports only k3 s2 p1 op1 (got k%d s%d p%d d%d)", who, d->ksize,
                d->stride, d->pad, d->dil);
  } else if (d->ksize == 1) {
    RCV_REQUIRE(d->stride == 1 && d->pad == 0 && d->dil == 1, RCV_ERR_UNSUPPORTED,
                "%s: 1x1 conv supports only s1 p0", who);
  } else {
    RCV_REQUIRE(d->ksize == 3, RCV_ERR_UNSUPPORTED, "%s: kernel size %d (supported 1, 3)", who, d->ksize);
    const bool ok = (d->stride == 1 && d->pad == 1 && d->dil == 1) ||
                    (d->stride == 1 && d->pad == 2 && d->dil == 2) ||
                    (d->stride == 2 && d->pad == 1 && d->dil == 1);
    RCV_REQUIRE(ok, RCV_ERR_UNSUPPORTED, "%s: 3x3 geometry s%d p%d d%d outside the hot path", who,
                d->stride, d->pad, d->dil);
  }
  RCV_REQUIRE(d->math >= RCV_MATH_FP32 && d->math <= RCV_MATH_BF16, RCV_ERR_BAD_ARG, "%s: bad math mode %d", who,
              d->math);
  RCV_REQUIRE(d->res_channels >= 0 && d->res_channels <= d->Cout, RCV_ERR_BAD_ARG, "%s: res_channels %d outside [0, %d]",
              who, d->res_channels, d->Cout);
  return RCV_OK;
}

void out_hw(const rcv_conv_desc* d, int* Ho, int* Wo) {
  if (d->transposed) {
    *Ho = 2 * d->H;
    *Wo = 2 * d->W;
  } else {
    *Ho = (d->H + 2 * d->pad - d->dil * (d->ksize - 1) - 1) / d->stride + 1;
    *Wo = (d->W + 2 * d->pad - d->dil * (d->ksize - 1) - 1) / d->stride + 1;
  }
}

// taps of an ordinary (cross-correlation) conv: input offset ky*dil - pad
void conv_taps(const rcv_conv_desc* d, RcvTapSet* t) {
  t->n = d->ksize * d->ksize;
  for (int ky = 0; ky < d->ksize; ++ky)
    for (int kx = 0; kx < d->ksize; ++kx) {
      const int i = ky * d->ksize + kx;
      t->dy[i] = (int8_t)(ky * d->dil - d->pad);
      t->dx[i] = (int8_t)(kx * d->dil - d->pad);
      t->wi[i] = (int8_t)i;
    }
}

// taps of the stride-1 input gradient: dx[y] = sum_ky dy[y + pad - ky*dil] w[ky]
void flipped_taps(const rcv_conv_desc* d, RcvTapSet* t) {
  t->n = d->ksize * d->ksize;
  for (int ky = 0; ky < d->ksize; ++ky)
    for (int kx = 0; kx < d->ksize; ++kx) {
      const int i = ky * d->ksize + kx;
      t->dy[i] = (int8_t)(d->pad - ky * d->dil);
      t->dx[i] = (int8_t)(d->pad - kx * d->dil);
      t->wi[i] = (int8_t)i;
    }
}

// Parity classes of "fine[2i+a] += coarse[i + d] * w[k]" with fine = 2*coarse + k - 1
// (k3 s2 p1): a=0 -> (k=1, d=0); a=1 -> (k=0, d=+1), (k=2, d=0).
void parity_taps(RcvTapSet t[4]) {
  static const int nk[2] = {1, 2};
  static const int kk[2][2] = {{1, 1}, {0, 2}};
  static const int dd[2][2] = {{0, 0}, {1, 0}};
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      RcvTapSet* s = &t[a * 2 + b];
      s->n = 0;
      for (int iy = 0; iy < nk[a]; ++iy)
        for (int ix = 0; ix < nk[b]; ++ix) {
          s->dy[s->n] = (int8_t)dd[a][iy];
          s->dx[s->n] = (int8_t)dd[b][ix];
          s->wi[s->n] = (int8_t)(kk[a][iy] * 3 + kk[b][ix]);
          s->n++;
        }
    }
}

}  // namespace

extern "C" int rcv_conv_out_hw(const rcv_conv_desc* d, int32_t* Ho, int32_t* Wo) {
  int rc = validate(d, "rcv_conv_out_hw");
  if (rc) return rc;
  RCV_REQUIRE(Ho && Wo, RCV_ERR_BAD_ARG, "rcv_conv_out_hw: null output");
  int h, w;
  out_hw(d, &h, &w);
  *Ho = h;
  *Wo = w;
  return RCV_OK;
}

namespace {

// Implicit-GEMM problem of the forward pass (tensor pointers left NULL).
void fwd_problem(const rcv_conv_desc* d, RcvIgemm* pp) {
  RcvIgemm& p = *pp;
  memset(&p, 0, sizeof(p));
  int Ho, Wo;
  out_hw(d, &Ho, &Wo);
  p.N = d->N; p.CA = d->Cin; p.CB = d->Cout;
  p.Hin = d->H; p.Win = d->W; p.Hout = Ho; p.Wout = Wo;
  p.epilogue = d->epilogue;
  p.math = d->math;
  p.ws = d->workspace;
  p.ws_bytes = d->workspace_bytes;
  p.res_C = d->res_channels > 0 ? d->res_channels : d->Cout;
  const int kk = d->ksize * d->ksize;
  if (!d->transposed) {
    p.Hg = Ho; p.Wg = Wo; p.gs = d->stride; p.ostep = 1; p.nclass = 1;
    p.wsA = kk;            // weight (Cout, Cin, k, k): stride of the reduced channel (Cin)
    p.wsB = d->Cin * kk;   // stride of the output channel
    conv_taps(d, &p.taps[0]);
  } else {
    p.Hg = d->H; p.Wg = d->W; p.gs = 1; p.ostep = 2; p.nclass = 4;
    p.wsA = d->Cout * 9;   // weight (Cin, Cout, 3, 3)
    p.wsB = 9;
    parity_taps(p.taps);
  }
}

// Implicit-GEMM problem of the input gradient: reduces over Cout, produces Cin channels.
int dgrad_problem(const rcv_conv_desc* d, RcvIgemm* pp) {
  RcvIgemm& p = *pp;
  memset(&p, 0, sizeof(p));
  int Ho, Wo;
  out_hw(d, &Ho, &Wo);
  p.N = d->N; p.CA = d->Cout; p.CB = d->Cin;
  p.Hin = Ho; p.Win = Wo; p.Hout = d->H; p.Wout = d->W;
  p.epilogue = RCV_EPI_NONE;
  p.math = d->math;
  p.ws = d->workspace;
  p.ws_bytes = d->workspace_bytes;
  p.res_C = d->Cin;
  const int kk = d->ksize * d->ksize;
  if (d->transposed) {
    // dx[ci,i,j] = sum dy[co, 2i+ky-1, 2j+kx-1] * w[ci,co,ky,kx]: a stride-2 conv over dy
    p.Hg = d->H; p.Wg = d->W; p.gs = 2; p.ostep = 1; p.nclass = 1;
    p.wsA = 9;             // weight (Cin, Cout, 3, 3): reduced channel = Cout
    p.wsB = d->Cout * 9;
    rcv_conv_desc s2 = *d;
    s2.ksize = 3; s2.dil = 1; s2.pad = 1;
    conv_taps(&s2, &p.taps[0]);
  } else if (d->stride == 1) {
    p.Hg = d->H; p.Wg = d->W; p.gs = 1; p.ostep = 1; p.nclass = 1;
    p.wsA = d->Cin * kk;   // weight (Cout, Cin, k, k): reduced channel = Cout
    p.wsB = kk;
    flipped_taps(d, &p.taps[0]);
  } else {
    // stride-2 conv: the input gradient is a transposed conv = four parity classes
    RCV_REQUIRE((d->H & 1) == 0 && (d->W & 1) == 0, RCV_ERR_UNSUPPORTED,
                "rcv_conv_dgrad: stride-2 conv needs even H, W (got %dx%d)", d->H, d->W);
    p.Hg = Ho; p.Wg = Wo; p.gs = 1; p.ostep = 2; p.nclass = 4;
    p.wsA = d->Cin * 9;
    p.wsB = 9;
    parity_taps(p.taps);
  }
  return RCV_OK;
}

int pack_problem(const rcv_conv_desc* d, int direction, RcvIgemm* p, const char* who) {
  int rc = validate(d, who);
  if (rc) return rc;
  RCV_REQUIRE(direction == RCV_PACK_FWD || direction == RCV_PACK_DGRAD, RCV_ERR_BAD_ARG,
              "%s: bad direction %d", who, direction);
  if (direction == RCV_PACK_FWD) {
    fwd_problem(d, p);
    return RCV_OK;
  }
  return dgrad_problem(d, p);
}

}  // namespace

extern "C" size_t rcv_conv_packed_bytes(const rcv_conv_desc* d, int direction) {
  RcvIgemm p;
  if (pack_problem(d, direction, &p, "rcv_conv_packed_bytes")) return 0;
  return rcv_umma_packed_bytes(p);
}

extern "C" int rcv_conv_uses_tensor_cores(const rcv_conv_desc* d, int direction) {
  RcvIgemm p;
  if (pack_problem(d, direction, &p, "rcv_conv_uses_tensor_cores")) return 0;
  return rcv_pick_engine(p, true) == RCV_ENGINE_UMMA ? 1 : 0;
}

extern "C" size_t rcv_conv_workspace_bytes(const rcv_conv_desc* d, int direction) {
  RcvIgemm p;
  if (pack_problem(d, direction, &p, "rcv_conv_workspace_bytes")) return 0;
  if (rcv_pick_engine(p, true) != RCV_ENGINE_UMMA) return 0;
  return rcv_umma_workspace_bytes(p);
}

namespace {
void wgrad_problem(const rcv_conv_desc* d, RcvWgrad* pp);
}

// Programmatic dependent launch for every kernel (rcv_common.cuh: rcv_launch / rcv_pdl_enter): RCV_PDL in the
// environment, else off, until rcv_set_pdl says otherwise.
static int g_pdl = -1;
bool rcv_pdl_enabled() {
  if (g_pdl < 0) {
    const char* e = getenv("RCV_PDL");
    g_pdl = (e && atoi(e) != 0) ? 1 : 0;
  }
  return g_pdl != 0;
}

extern "C" int rcv_set_pdl(int on) {
  const int prev = rcv_pdl_enabled() ? 1 : 0;
  g_pdl = on ? 1 : 0;
  return prev;
}

extern "C" int rcv_get_pdl(void) { return rcv_pdl_enabled() ? 1 : 0; }

extern "C" int rcv_conv_engine(const rcv_conv_desc* d, int direction) {
  if (direction == RCV_DIR_WGRAD) {
    int rc = validate(d, "rcv_conv_engine");
    if (rc) return rc;
    RcvWgrad w;
    wgrad_problem(d, &w);
    return rcv_pick_wgrad_engine(w);
  }
  RcvIgemm p;
  int rc = pack_problem(d, direction, &p, "rcv_conv_engine");
  if (rc) return rc;
  return rcv_pick_engine(p, true);
}

extern "C" int rcv_conv_pack(const rcv_conv_desc* d, int direction, const float* w, void* packed,
                             void* stream) {
  RcvIgemm p;
  int rc = pack_problem(d, direction, &p, "rcv_conv_pack");
  if (rc) return rc;
  RCV_REQUIRE(w && packed, RCV_ERR_BAD_ARG, "rcv_conv_pack: null tensor");
  p.w = w;
  return rcv_launch_umma_pack(p, packed, (cudaStream_t)stream);
}

extern "C" size_t rcv_conv_pack_table_bytes(int32_t njobs) {
  return njobs > 0 ? (size_t)njobs * sizeof(RcvPackJob) : 0;
}

extern "C" int rcv_conv_pack_table_build(int32_t njobs, const rcv_conv_desc* descs, const int32_t* directions,
                                         const float* const* weights, void* const* packed, void* host_table,
                                         int64_t* total_chunks) {
  RCV_REQUIRE(njobs >= 1 && njobs <= RCV_PACK_MAX_JOBS, RCV_ERR_BAD_ARG, "pack table: %d jobs (1..%d)", njobs,
              RCV_PACK_MAX_JOBS);
  RCV_REQUIRE(descs && directions && weights && packed && host_table && total_chunks, RCV_ERR_BAD_ARG,
              "pack table: null argument");
  RcvPackJob* jobs = reinterpret_cast<RcvPackJob*>(host_table);
  long long begin = 0;
  for (int j = 0; j < njobs; ++j) {
    RcvIgemm p;
    int rc = pack_problem(&descs[j], directions[j], &p, "rcv_conv_pack_table_build");
    if (rc) return rc;
    RCV_REQUIRE(weights[j] && packed[j], RCV_ERR_BAD_ARG, "pack table: null tensor in job %d", j);
    p.w = weights[j];
    rc = rcv_umma_pack_job(p, packed[j], begin, &jobs[j]);
    if (rc) return rc;
    begin += jobs[j].chunks;
  }
  *total_chunks = begin;
  return RCV_OK;
}

extern "C" int rcv_conv_pack_table_run(const void* device_table, int32_t njobs, int64_t total_chunks, void* stream) {
  RCV_REQUIRE(device_table != nullptr, RCV_ERR_BAD_ARG, "pack table: null device table");
  return rcv_launch_umma_pack_multi(reinterpret_cast<const RcvPackJob*>(device_table), njobs, total_chunks,
                                    (cudaStream_t)stream);
}

static int conv_fwd_impl(const rcv_conv_desc* d, const float* x, const float* in_scale, const float* in_shift,
                         int in_relu, const float* w, const void* wpacked, const float* bias, const float* scale,
                         const float* shift, const float* residual, float* y, double* stats, void* stream);

extern "C" int rcv_conv_fwd(const rcv_conv_desc* d, const float* x, const float* w, const void* wpacked,
                            const float* bias, const float* scale, const float* shift,
                            const float* residual, float* y, double* stats, void* stream) {
  return conv_fwd_impl(d, x, nullptr, nullptr, 0, w, wpacked, bias, scale, shift, residual, y, stats, stream);
}

extern "C" int rcv_conv_normalises_on_load(const rcv_conv_desc* d) {
  RcvIgemm p;
  if (pack_problem(d, RCV_PACK_FWD, &p, "rcv_conv_normalises_on_load")) return 0;
  if (rcv_pick_engine(p, true) != RCV_ENGINE_UMMA) return 0;
  return rcv_umma_takes_input_transform(p) ? 1 : 0;
}

extern "C" int rcv_conv_fwd_nl(const rcv_conv_desc* d, const float* x, const float* in_scale, const float* in_shift,
                               int in_relu, const float* w, const void* wpacked, const float* bias,
                               const float* scale, const float* shift, const float* residual, float* y,
                               double* stats, void* stream) {
  RCV_REQUIRE(in_scale && in_shift, RCV_ERR_BAD_ARG, "rcv_conv_fwd_nl: null input scale / shift");
  RCV_REQUIRE(rcv_conv_normalises_on_load(d), RCV_ERR_UNSUPPORTED,
              "rcv_conv_fwd_nl: this layer does not run on the halo-staged tensor-core kernel "
              "(query rcv_conv_normalises_on_load first)");
  return conv_fwd_impl(d, x, in_scale, in_shift, in_relu, w, wpacked, bias, scale, shift, residual, y, stats, stream);
}

static int conv_fwd_impl(const rcv_conv_desc* d, const float* x, const float* in_scale, const float* in_shift,
                         int in_relu, const float* w, const void* wpacked, const float* bias, const float* scale,
                         const float* shift, const float* residual, float* y, double* stats, void* stream) {
  int rc = validate(d, "rcv_conv_fwd");
  if (rc) return rc;
  RCV_REQUIRE(x && w && y, RCV_ERR_BAD_ARG, "rcv_conv_fwd: null tensor");
  RCV_REQUIRE(d->epilogue >= RCV_EPI_NONE && d->epilogue <= RCV_EPI_AFFINE, RCV_ERR_BAD_ARG,
              "rcv_conv_fwd: bad epilogue %d", d->epilogue);
  const bool needs_affine = d->epilogue == RCV_EPI_RELU_AFFINE || d->epilogue == RCV_EPI_AFFINE_RELU ||
                            d->epilogue == RCV_EPI_AFFINE;
  RCV_REQUIRE(!needs_affine || (scale && shift), RCV_ERR_BAD_ARG,
              "rcv_conv_fwd: affine epilogue needs scale and shift");
  RcvIgemm p;
  fwd_problem(d, &p);
  RCV_REQUIRE(p.Hout > 0 && p.Wout > 0, RCV_ERR_BAD_ARG, "rcv_conv_fwd: empty output");
  p.in = x; p.w = w; p.wpacked = wpacked; p.out = y; p.bias = bias; p.scale = scale; p.shift = shift;
  p.residual = residual; p.stats = stats;
  p.in_scale = in_scale; p.in_shift = in_shift; p.in_relu = in_relu;
  return rcv_launch_igemm(p, (cudaStream_t)stream);
}

extern "C" int rcv_conv_dgrad(const rcv_conv_desc* d, const float* dy, const float* w, const void* wpacked,
                              const float* residual, float* dx, void* stream) {
  int rc = validate(d, "rcv_conv_dgrad");
  if (rc) return rc;
  RCV_REQUIRE(dy && w && dx, RCV_ERR_BAD_ARG, "rcv_conv_dgrad: null tensor");
  RcvIgemm p;
  rc = dgrad_problem(d, &p);
  if (rc) return rc;
  p.in = dy; p.w = w; p.wpacked = wpacked; p.out = dx;
  p.residual = residual;
  return rcv_launch_igemm(p, (cudaStream_t)stream);
}

namespace {
// Pixel-reduction problem of the weight gradient (tensor pointers left NULL; dbias handled by the caller).
void wgrad_problem(const rcv_conv_desc* d, RcvWgrad* pp) {
  RcvWgrad& p = *pp;
  memset(&p, 0, sizeof(p));
  int Ho, Wo;
  out_hw(d, &Ho, &Wo);
  p.math = d->math;
  p.N = d->N;
  const int kk = d->ksize * d->ksize;
  if (!d->transposed) {
    p.CA = d->Cin; p.CB = d->Cout;
    p.Hin = d->H; p.Win = d->W; p.Hg = Ho; p.Wg = Wo; p.gs = d->stride;
    p.wsA = kk; p.wsB = d->Cin * kk;
    conv_taps(d, &p.taps);
  } else {
    // dw[ci,co,ky,kx] = sum x[ci,i,j] * dy[co, 2i+ky-1, 2j+kx-1]
    p.CA = d->Cout; p.CB = d->Cin;
    p.Hin = Ho; p.Win = Wo; p.Hg = d->H; p.Wg = d->W; p.gs = 2;
    p.wsA = 9; p.wsB = d->Cout * 9;
    rcv_conv_desc s2 = *d;
    conv_taps(&s2, &p.taps);
  }
}
}  // namespace

extern "C" int rcv_conv_wgrad_normalises_on_load(const rcv_conv_desc* d) {
  if (validate(d, "rcv_conv_wgrad_normalises_on_load") || d->transposed) return 0;
  RcvWgrad p;
  wgrad_problem(d, &p);
  return (rcv_pick_wgrad_engine(p) == RCV_ENGINE_UMMA && rcv_umma_wgrad_takes_input_transform(p)) ? 1 : 0;
}

static int conv_wgrad_impl(const rcv_conv_desc* d, const float* x, const float* in_scale, const float* in_shift,
                           int in_relu, const float* dy, float* dw, float* dbias, void* stream);

extern "C" int rcv_conv_wgrad(const rcv_conv_desc* d, const float* x, const float* dy, float* dw,
                              float* dbias, void* stream) {
  return conv_wgrad_impl(d, x, nullptr, nullptr, 0, dy, dw, dbias, stream);
}

extern "C" int rcv_conv_wgrad_nl(const rcv_conv_desc* d, const float* x, const float* in_scale, const float* in_shift,
                                 int in_relu, const float* dy, float* dw, float* dbias, void* stream) {
  RCV_REQUIRE(in_scale && in_shift, RCV_ERR_BAD_ARG, "rcv_conv_wgrad_nl: null input scale / shift");
  RCV_REQUIRE(rcv_conv_wgrad_normalises_on_load(d), RCV_ERR_UNSUPPORTED,
              "rcv_conv_wgrad_nl: this layer's weight gradient does not run on the tensor-core quad-gather kernel "
              "(query rcv_conv_wgrad_normalises_on_load first)");
  return conv_wgrad_impl(d, x, in_scale, in_shift, in_relu, dy, dw, dbias, stream);
}

static int conv_wgrad_impl(const rcv_conv_desc* d, const float* x, const float* in_scale, const float* in_shift,
                           int in_relu, const float* dy, float* dw, float* dbias, void* stream) {
  int rc = validate(d, "rcv_conv_wgrad");
  if (rc) return rc;
  RCV_REQUIRE(x && dy && dw, RCV_ERR_BAD_ARG, "rcv_conv_wgrad: null tensor");
  RcvWgrad p;
  wgrad_problem(d, &p);
  p.dw = dw;
  p.in_scale = in_scale; p.in_shift = in_shift; p.in_relu = in_relu;
  if (!d->transposed) {
    p.src = x; p.row = dy; p.dbias = dbias;
  } else {
    p.src = dy; p.row = x; p.dbias = nullptr;
    if (dbias) {
      rc = rcv_channel_sum(d->N, d->Cout, (int64_t)p.Hin * p.Win, dy, dbias, stream);
      if (rc) return rc;
    }
  }
  return rcv_launch_wgrad(p, (cudaStream_t)stream);
}
