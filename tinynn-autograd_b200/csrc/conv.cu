// NHWC convolution and max-pooling passes (new: no reference counterpart).  Conv2D is lowered to
// im2col + the existing GEMM route (core/layers.py); these are the memory-bound passes around it.
//
// Every kernel here is one launch, indexes in int64, moves EL consecutive channels per thread as
// one 16-byte access when C and the pointers allow it, and uses no atomics: each output element is
// written by exactly one thread, and the backward passes are GATHERS that sum their contributions
// in a fixed order, so results are bit-reproducible run to run and under graph replay.
#include "common.cuh"

namespace tnn {

struct Geom {
  int64_t N, H, W, C;   // input (NHWC)
  int64_t KH, KW;       // window
  int64_t SH, SW;       // stride
  int64_t PH0, PW0;     // padding before the first row / column
  int64_t OH, OW;       // output rows / columns
};

// col[(n,oh,ow), (kh,kw,c)] = x[n, oh*SH + kh - PH0, ow*SW + kw - PW0, c], 0 outside the image.
// One thread per EL-vector of col, in col's row-major order: the stores are fully coalesced.
template <typename T, int EL>
__global__ void __launch_bounds__(256) im2col_kernel(T* __restrict__ col, const T* __restrict__ x, Geom g) {
  using P = Pack<T, EL>;
  const int64_t Cv = g.C / EL;
  const int64_t n_vec = g.N * g.OH * g.OW * g.KH * g.KW * Cv;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  P* __restrict__ out = reinterpret_cast<P*>(col);
  const P* __restrict__ in = reinterpret_cast<const P*>(x);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
    int64_t r = i;
    const int64_t cv = r % Cv;
    r /= Cv;
    const int64_t kw = r % g.KW;
    r /= g.KW;
    const int64_t kh = r % g.KH;
    r /= g.KH;
    const int64_t ow = r % g.OW;
    r /= g.OW;
    const int64_t oh = r % g.OH;
    const int64_t n = r / g.OH;
    const int64_t ih = oh * g.SH + kh - g.PH0;
    const int64_t iw = ow * g.SW + kw - g.PW0;
    P v{};
    if (ih >= 0 && ih < g.H && iw >= 0 && iw < g.W) v = in[((n * g.H + ih) * g.W + iw) * Cv + cv];
    out[i] = v;
  }
}

// dx[n,ih,iw,c] = sum over the (kh, kw) whose window position reads (ih, iw), in ascending (kh, kw)
// order, of dcol[(n,oh,ow), (kh,kw,c)].  One thread per EL-vector of dx; dx is written, not
// accumulated into.
template <typename T, int EL>
__global__ void __launch_bounds__(256) col2im_kernel(T* __restrict__ dx, const T* __restrict__ dcol, Geom g) {
  using P = Pack<T, EL>;
  const int64_t Cv = g.C / EL;
  const int64_t n_vec = g.N * g.H * g.W * Cv;
  const int64_t row_v = g.KH * g.KW * Cv;   // one col row, in vectors
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  P* __restrict__ out = reinterpret_cast<P*>(dx);
  const P* __restrict__ in = reinterpret_cast<const P*>(dcol);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
    int64_t r = i;
    const int64_t cv = r % Cv;
    r /= Cv;
    const int64_t iw = r % g.W;
    r /= g.W;
    const int64_t ih = r % g.H;
    const int64_t n = r / g.H;
    // the windows oh that read row ih: oh*SH - PH0 <= ih <= oh*SH - PH0 + KH - 1, kh = th - oh*SH;
    // walking oh downwards walks kh upwards (same for the columns)
    const int64_t th = ih + g.PH0, tw = iw + g.PW0;
    const int64_t oh_hi = min(th / g.SH, g.OH - 1);
    const int64_t ow_hi = min(tw / g.SW, g.OW - 1);
    const int64_t oh_lo = th - g.KH + 1 <= 0 ? 0 : ceil_div(th - g.KH + 1, g.SH);
    const int64_t ow_lo = tw - g.KW + 1 <= 0 ? 0 : ceil_div(tw - g.KW + 1, g.SW);
    P acc{};
    for (int64_t oh = oh_hi; oh >= oh_lo; --oh) {
      const int64_t kh = th - oh * g.SH;
      for (int64_t ow = ow_hi; ow >= ow_lo; --ow) {
        const int64_t kw = tw - ow * g.SW;
        const P d = in[((n * g.OH + oh) * g.OW + ow) * row_v + (kh * g.KW + kw) * Cv + cv];
#pragma unroll
        for (int e = 0; e < EL; ++e) acc.v[e] += d.v[e];
      }
    }
    out[i] = acc;
  }
}

// y[n,oh,ow,c] = max over the real (unpadded) elements of the window, arg = the window offset
// kh*KW + kw of the one selected: the first in row-major window order among the maxima, or the
// first NaN (np.max / np.argmax over the flattened window).  SAME padding leaves at least one real
// element in every window, so the first real element seeds the search.
template <typename T, int EL>
__global__ void __launch_bounds__(256)
maxpool_fwd_kernel(T* __restrict__ y, int32_t* __restrict__ arg, const T* __restrict__ x, Geom g) {
  using P = Pack<T, EL>;
  using I = Pack<int32_t, EL>;
  const int64_t Cv = g.C / EL;
  const int64_t n_vec = g.N * g.OH * g.OW * Cv;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const P* __restrict__ in = reinterpret_cast<const P*>(x);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
    int64_t r = i;
    const int64_t cv = r % Cv;
    r /= Cv;
    const int64_t ow = r % g.OW;
    r /= g.OW;
    const int64_t oh = r % g.OH;
    const int64_t n = r / g.OH;
    const int64_t h0 = oh * g.SH - g.PH0, w0 = ow * g.SW - g.PW0;
    P best{};
    I sel{};
    bool seeded = false;
    for (int64_t kh = 0; kh < g.KH; ++kh) {
      const int64_t ih = h0 + kh;
      if (ih < 0 || ih >= g.H) continue;
      for (int64_t kw = 0; kw < g.KW; ++kw) {
        const int64_t iw = w0 + kw;
        if (iw < 0 || iw >= g.W) continue;
        const P v = in[((n * g.H + ih) * g.W + iw) * Cv + cv];
        const int32_t k = (int32_t)(kh * g.KW + kw);
#pragma unroll
        for (int e = 0; e < EL; ++e) {
          const T b = best.v[e], c = v.v[e];
          // b != b: the window already holds a NaN, which stays selected
          if (!seeded || (b == b && (c != c || c > b))) {
            best.v[e] = c;
            sel.v[e] = k;
          }
        }
        seeded = true;
      }
    }
    reinterpret_cast<P*>(y)[i] = best;
    reinterpret_cast<I*>(arg)[i] = sel;
  }
}

// dx[n,ih,iw,c] = sum, over the windows (oh ascending, then ow) that cover (ih, iw) and selected it,
// of dy[n,oh,ow,c].  Covers overlapping (stride < window) and disjoint windows alike.
template <typename T, int EL>
__global__ void __launch_bounds__(256) maxpool_bwd_kernel(T* __restrict__ dx, const T* __restrict__ dy,
                                                          const int32_t* __restrict__ arg, Geom g) {
  using P = Pack<T, EL>;
  using I = Pack<int32_t, EL>;
  const int64_t Cv = g.C / EL;
  const int64_t n_vec = g.N * g.H * g.W * Cv;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const P* __restrict__ gin = reinterpret_cast<const P*>(dy);
  const I* __restrict__ ain = reinterpret_cast<const I*>(arg);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += stride) {
    int64_t r = i;
    const int64_t cv = r % Cv;
    r /= Cv;
    const int64_t iw = r % g.W;
    r /= g.W;
    const int64_t ih = r % g.H;
    const int64_t n = r / g.H;
    // windows oh with oh*SH - PH0 <= ih <= oh*SH - PH0 + KH - 1
    const int64_t th = ih + g.PH0, tw = iw + g.PW0;
    const int64_t oh_hi = min(th / g.SH, g.OH - 1);
    const int64_t ow_hi = min(tw / g.SW, g.OW - 1);
    const int64_t oh_lo = th - g.KH + 1 <= 0 ? 0 : ceil_div(th - g.KH + 1, g.SH);
    const int64_t ow_lo = tw - g.KW + 1 <= 0 ? 0 : ceil_div(tw - g.KW + 1, g.SW);
    P acc{};
    for (int64_t oh = oh_lo; oh <= oh_hi; ++oh) {
      const int64_t kh = th - oh * g.SH;
      for (int64_t ow = ow_lo; ow <= ow_hi; ++ow) {
        const int32_t k = (int32_t)(kh * g.KW + (tw - ow * g.SW));
        const int64_t o = ((n * g.OH + oh) * g.OW + ow) * Cv + cv;
        const I a = ain[o];
        const P d = gin[o];
#pragma unroll
        for (int e = 0; e < EL; ++e)
          if (a.v[e] == k) acc.v[e] += d.v[e];
      }
    }
    reinterpret_cast<P*>(dx)[i] = acc;
  }
}

static int check_geom(const char* name, const Geom& g) {
  if (g.N < 0 || g.H < 0 || g.W < 0 || g.C <= 0 || g.KH <= 0 || g.KW <= 0 || g.SH <= 0 || g.SW <= 0 ||
      g.PH0 < 0 || g.PW0 < 0 || g.PH0 >= g.KH || g.PW0 >= g.KW || g.OH < 0 || g.OW < 0)
    TNN_FAIL(std::string(name) + ": bad geometry");
  // every output window must lie within the padded image: (O-1)*S + K <= P0 + I + (K-1)
  if ((g.OH > 0 && (g.OH - 1) * g.SH - g.PH0 >= g.H) || (g.OW > 0 && (g.OW - 1) * g.SW - g.PW0 >= g.W))
    TNN_FAIL(std::string(name) + ": output extent exceeds the padded input");
  // (the int32 window offsets of the pooling passes)
  if (g.KH * g.KW > INT32_MAX) TNN_FAIL(std::string(name) + ": window too large");
  return 0;
}

// Launches f(T{}, std::integral_constant<int, EL>{}, grid) over n elements: EL = 16 / sizeof(T) when C
// is a multiple of it and every pointer is 16-byte aligned, EL = 1 otherwise
template <typename F>
static int launch_vec(const char* name, int dtype, bool ptrs_aligned, const Geom& g, int64_t n, F&& f) {
  return with_float_type(dtype, name, [&](auto tag) {
    constexpr int V = 16 / sizeof(tag);
    const bool vec = ptrs_aligned && g.C % V == 0;
    const int64_t work = vec ? n / V : n;
    if (work == 0) return 0;
    const int grid = ew_grid(work, 256);
    with_bool(vec, [&](auto v) { f(tag, std::integral_constant<int, v ? V : 1>{}, grid); });
    TNN_POST_LAUNCH();
    return 0;
  });
}

static Geom make_geom(int64_t N, int64_t H, int64_t W, int64_t C, int64_t KH, int64_t KW, int64_t SH,
                      int64_t SW, int64_t PH0, int64_t PW0, int64_t OH, int64_t OW) {
  Geom g;
  g.N = N, g.H = H, g.W = W, g.C = C, g.KH = KH, g.KW = KW, g.SH = SH, g.SW = SW;
  g.PH0 = PH0, g.PW0 = PW0, g.OH = OH, g.OW = OW;
  return g;
}

}  // namespace tnn

using namespace tnn;

extern "C" {

int tnn_im2col(int dtype, void* col, const void* x, int64_t N, int64_t H, int64_t W, int64_t C, int64_t KH,
               int64_t KW, int64_t SH, int64_t SW, int64_t PH0, int64_t PW0, int64_t OH, int64_t OW) {
  TNN_REQUIRE_INIT();
  const Geom g = make_geom(N, H, W, C, KH, KW, SH, SW, PH0, PW0, OH, OW);
  if (check_geom("tnn_im2col", g)) return 1;
  return launch_vec("tnn_im2col", dtype, aligned16(col) && aligned16(x), g, N * OH * OW * KH * KW * C,
                    [&](auto tag, auto EL, int grid) {
                      using T = decltype(tag);
                      im2col_kernel<T, EL><<<grid, 256, 0, ctx().stream>>>((T*)col, (const T*)x, g);
                    });
}

int tnn_col2im(int dtype, void* dx, const void* dcol, int64_t N, int64_t H, int64_t W, int64_t C, int64_t KH,
               int64_t KW, int64_t SH, int64_t SW, int64_t PH0, int64_t PW0, int64_t OH, int64_t OW) {
  TNN_REQUIRE_INIT();
  const Geom g = make_geom(N, H, W, C, KH, KW, SH, SW, PH0, PW0, OH, OW);
  if (check_geom("tnn_col2im", g)) return 1;
  return launch_vec("tnn_col2im", dtype, aligned16(dx) && aligned16(dcol), g, N * H * W * C,
                    [&](auto tag, auto EL, int grid) {
                      using T = decltype(tag);
                      col2im_kernel<T, EL><<<grid, 256, 0, ctx().stream>>>((T*)dx, (const T*)dcol, g);
                    });
}

int tnn_maxpool_fwd(int dtype, void* y, int32_t* arg, const void* x, int64_t N, int64_t H, int64_t W,
                    int64_t C, int64_t PH, int64_t PW, int64_t SH, int64_t SW, int64_t PH0, int64_t PW0,
                    int64_t OH, int64_t OW) {
  TNN_REQUIRE_INIT();
  const Geom g = make_geom(N, H, W, C, PH, PW, SH, SW, PH0, PW0, OH, OW);
  if (check_geom("tnn_maxpool_fwd", g)) return 1;
  return launch_vec("tnn_maxpool_fwd", dtype, aligned16(y) && aligned16(arg) && aligned16(x), g, N * OH * OW * C,
                    [&](auto tag, auto EL, int grid) {
                      using T = decltype(tag);
                      maxpool_fwd_kernel<T, EL><<<grid, 256, 0, ctx().stream>>>((T*)y, arg, (const T*)x, g);
                    });
}

int tnn_maxpool_bwd(int dtype, void* dx, const void* dy, const int32_t* arg, int64_t N, int64_t H, int64_t W,
                    int64_t C, int64_t PH, int64_t PW, int64_t SH, int64_t SW, int64_t PH0, int64_t PW0,
                    int64_t OH, int64_t OW) {
  TNN_REQUIRE_INIT();
  const Geom g = make_geom(N, H, W, C, PH, PW, SH, SW, PH0, PW0, OH, OW);
  if (check_geom("tnn_maxpool_bwd", g)) return 1;
  return launch_vec("tnn_maxpool_bwd", dtype, aligned16(dx) && aligned16(dy) && aligned16(arg), g, N * H * W * C,
                    [&](auto tag, auto EL, int grid) {
                      using T = decltype(tag);
                      maxpool_bwd_kernel<T, EL><<<grid, 256, 0, ctx().stream>>>((T*)dx, (const T*)dy, arg, g);
                    });
}

}  // extern "C"
