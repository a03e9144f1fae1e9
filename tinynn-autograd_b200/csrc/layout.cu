// Layout kernels: ops.py:268-279 (transpose_), 282-290 (getitem_ and its assignment-style
// backward), 312-321 (pad_ and its slice backward).  Reshape/flatten (ops.py:302-309, 324-330)
// are views on the host side and never reach this file.
#include <algorithm>

#include "common.cuh"

namespace tnn {

struct CopyArgs {
  int ndim;
  int64_t shape[TNN_MAX_DIMS];
  int64_t ds[TNN_MAX_DIMS];
  int64_t ss[TNN_MAX_DIMS];
};

// one thread per element of the index space; the innermost collapsed axis is walked by
// consecutive threads so whichever side has unit stride there is coalesced
template <typename T>
__global__ void __launch_bounds__(256)
strided_copy_kernel(T* dst, const T* src, int64_t n, CopyArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    int64_t rem = i, so = 0, d_o = 0;
#pragma unroll 1
    for (int d = a.ndim - 1; d >= 0; --d) {
      int64_t q = rem / a.shape[d];
      int64_t c = rem - q * a.shape[d];
      rem = q;
      so += c * a.ss[d];
      d_o += c * a.ds[d];
    }
    dst[d_o] = src[so];
  }
}

// 2-D transpose through shared memory (both sides coalesced): dst[c*ldd + r] = src[r*lds + c]
template <typename T>
__global__ void __launch_bounds__(256)
transpose2d_kernel(T* dst, const T* src, int64_t R, int64_t C, int64_t lds, int64_t ldd) {
  __shared__ T tile[32][33];
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
  for (int j = 0; j < 32; j += 8) {
    int64_t r = r0 + ty + j, c = c0 + tx;
    if (r < R && c < C) tile[ty + j][tx] = src[r * lds + c];
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 32; j += 8) {
    int64_t c = c0 + ty + j, r = r0 + tx;
    if (r < R && c < C) dst[c * ldd + r] = tile[tx][ty + j];
  }
}

// rows: a warp moves one row with 128-bit accesses when the row is 16-byte sized and aligned
template <typename T, bool GATHER>
__global__ void __launch_bounds__(256)
rows_kernel(T* out, const T* in, const int64_t* idx, int64_t n_idx, int64_t row_elems,
            int64_t n_rows_other, int vec_ok) {
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * 8;
  for (int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); i < n_idx; i += warps_total) {
    int64_t j = idx[i];
    if (j < 0) j += n_rows_other;          // numpy negative indices
    if (j < 0 || j >= n_rows_other) continue;  // bounds are validated on the host
    const T* s = GATHER ? in + j * row_elems : in + i * row_elems;
    T* d = GATHER ? out + i * row_elems : out + j * row_elems;
    if (vec_ok) {
      const int64_t nv = row_elems * sizeof(T) / 16;
      const int4* s4 = reinterpret_cast<const int4*>(s);
      int4* d4 = reinterpret_cast<int4*>(d);
      for (int64_t k = lane; k < nv; k += 32) d4[k] = s4[k];
    } else {
      for (int64_t k = lane; k < row_elems; k += 32) d[k] = s[k];
    }
  }
}

template <typename T, bool GATHER>
__global__ void __launch_bounds__(256)
flat_index_kernel(T* out, const T* in, const int64_t* idx, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (GATHER) out[i] = in[idx[i]];
    else out[idx[i]] = in[i];
  }
}

template <typename T>
static int strided_copy_impl(T* dst, const T* src, int ndim, const int64_t* shape,
                             const int64_t* ds, const int64_t* ss) {
  // collapse axes that nest on both sides
  CopyArgs a;
  int nd = 0;
  int64_t total = 1;
  for (int d = 0; d < ndim; ++d) total *= shape[d];
  if (total == 0) return 0;
  for (int d = 0; d < ndim; ++d) {
    if (shape[d] == 1) continue;
    if (nd > 0 && a.ds[nd - 1] == ds[d] * shape[d] && a.ss[nd - 1] == ss[d] * shape[d]) {
      a.shape[nd - 1] *= shape[d];
      a.ds[nd - 1] = ds[d];
      a.ss[nd - 1] = ss[d];
    } else {
      a.shape[nd] = shape[d];
      a.ds[nd] = ds[d];
      a.ss[nd] = ss[d];
      ++nd;
    }
  }
  if (nd == 0) {
    nd = 1;
    a.shape[0] = 1;
    a.ds[0] = a.ss[0] = 1;
  }
  a.ndim = nd;
  for (int d = nd; d < TNN_MAX_DIMS; ++d) {
    a.shape[d] = 1;
    a.ds[d] = a.ss[d] = 0;
  }
  cudaStream_t st = ctx().stream;
  // pure 2-D transpose: (R, C) index space, src row-major, dst column-major (or vice versa)
  if (nd == 2 && a.ss[1] == 1 && a.ds[0] == 1 && a.shape[0] >= 32 && a.shape[1] >= 32) {
    dim3 grid((unsigned)ceil_div(a.shape[1], 32), (unsigned)ceil_div(a.shape[0], 32));
    if (grid.y <= 65535) {
      transpose2d_kernel<T><<<grid, 256, 0, st>>>(dst, src, a.shape[0], a.shape[1], a.ss[0], a.ds[1]);
      TNN_POST_LAUNCH();
      return 0;
    }
  }
  int grid = ew_grid(total, 256);
  strided_copy_kernel<T><<<grid, 256, 0, st>>>(dst, src, total, a);
  TNN_POST_LAUNCH();
  return 0;
}

// dense one-hot rows from integer class labels (examples/mnist/run.py:27-28 get_one_hot, done on
// the device so a host-fed batch ships 4 B per sample instead of 4*C): out[r, c] = (labels[r] == c).
// A label outside [0, C) gives an all-zero row.
template <typename T>
__global__ void __launch_bounds__(256)
one_hot_kernel(T* out, const int32_t* labels, int64_t B, int64_t C) {
  const int64_t n = B * C;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int64_t r = i / C;
    out[i] = (int64_t)labels[r] == i - r * C ? T(1) : T(0);
  }
}

// float32 rows whose length is a multiple of 4: one 128-bit store per thread
__global__ void __launch_bounds__(256)
one_hot_vec_kernel(float4* out, const int32_t* labels, int64_t B, int64_t C4) {
  const int64_t n = B * C4;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int64_t r = i / C4;
    const int64_t c = (i - r * C4) * 4;
    const int64_t d = (int64_t)labels[r] - c;
    out[i] = make_float4(d == 0 ? 1.f : 0.f, d == 1 ? 1.f : 0.f, d == 2 ? 1.f : 0.f, d == 3 ? 1.f : 0.f);
  }
}

}  // namespace tnn

using namespace tnn;

extern "C" {

int tnn_strided_copy(int dtype, void* dst, const void* src, int ndim, const int64_t* shape,
                     const int64_t* dst_strides, const int64_t* src_strides) {
  TNN_REQUIRE_INIT();
  if (ndim < 0 || ndim > TNN_MAX_DIMS) TNN_FAIL("tnn_strided_copy: rank above TNN_MAX_DIMS");
  return with_float_type(dtype, "tnn_strided_copy", [&](auto tag) {
    using T = decltype(tag);
    return strided_copy_impl<T>((T*)dst, (const T*)src, ndim, shape, dst_strides, src_strides);
  });
}

static int rows_common(bool gather, int dtype, void* out, const void* in, const int64_t* idx,
                       int64_t n_idx, int64_t row_elems, int64_t n_rows_other) {
  TNN_REQUIRE_INIT();
  if (n_idx <= 0 || row_elems <= 0) return 0;
  return with_float_type(dtype, gather ? "tnn_gather_rows" : "tnn_scatter_rows", [&](auto tag) {
    using T = decltype(tag);
    const int vec_ok = (row_elems * sizeof(T)) % 16 == 0 && aligned16(out) && aligned16(in);
    const int grid = (int)std::min<int64_t>(ceil_div(n_idx, 8), (int64_t)ctx().sm_count * 16);
    with_bool(gather, [&](auto G) {
      rows_kernel<T, G><<<grid, 256, 0, ctx().stream>>>((T*)out, (const T*)in, idx, n_idx, row_elems, n_rows_other,
                                                        vec_ok);
    });
    TNN_POST_LAUNCH();
    return 0;
  });
}

int tnn_gather_rows(int dtype, void* out, const void* x, const int64_t* idx_dev, int64_t n_idx,
                    int64_t row_elems, int64_t n_rows_src) {
  return rows_common(true, dtype, out, x, idx_dev, n_idx, row_elems, n_rows_src);
}

int tnn_scatter_rows(int dtype, void* out, const void* g, const int64_t* idx_dev, int64_t n_idx,
                     int64_t row_elems, int64_t n_rows_dst) {
  return rows_common(false, dtype, out, g, idx_dev, n_idx, row_elems, n_rows_dst);
}

static int flat_common(bool gather, int dtype, void* out, const void* in, const int64_t* idx,
                       int64_t n) {
  TNN_REQUIRE_INIT();
  if (n <= 0) return 0;
  return with_float_type(dtype, gather ? "tnn_gather_flat" : "tnn_scatter_flat", [&](auto tag) {
    using T = decltype(tag);
    with_bool(gather, [&](auto G) {
      flat_index_kernel<T, G><<<ew_grid(n, 256), 256, 0, ctx().stream>>>((T*)out, (const T*)in, idx, n);
    });
    TNN_POST_LAUNCH();
    return 0;
  });
}

int tnn_gather_flat(int dtype, void* out, const void* x, const int64_t* idx_dev, int64_t n) {
  return flat_common(true, dtype, out, x, idx_dev, n);
}

int tnn_scatter_flat(int dtype, void* out, const void* g, const int64_t* idx_dev, int64_t n) {
  return flat_common(false, dtype, out, g, idx_dev, n);
}

int tnn_one_hot(int dtype, void* out, const int32_t* labels_dev, int64_t B, int64_t C) {
  TNN_REQUIRE_INIT();
  if (B <= 0 || C <= 0) return 0;
  return with_float_type(dtype, "tnn_one_hot", [&](auto tag) {
    using T = decltype(tag);
    cudaStream_t st = ctx().stream;
    if (std::is_same<T, float>::value && C % 4 == 0 && aligned16(out))
      one_hot_vec_kernel<<<ew_grid(B * (C / 4), 256), 256, 0, st>>>((float4*)out, labels_dev, B, C / 4);
    else
      one_hot_kernel<T><<<ew_grid(B * C, 256), 256, 0, st>>>((T*)out, labels_dev, B, C);
    TNN_POST_LAUNCH();
    return 0;
  });
}

}  // extern "C"
