// Convolution trunk of the CNN head (jorldy/core/network/head.py:21-61: x/255 -> conv 8x8 s4 ->
// 4x4 s2 -> 3x3 s1, ReLU each, flatten in C,H,W order) lowered to the shared fp32 GEMM:
//   forward   col = im2col(x)  [B*OH*OW, C*KH*KW]   then  y = relu(col W^T + b)   (jb_gemm, NHWC out)
//   backward  dW = dy^T col ; dcol = dy W ; dx = col2im(dcol)  (gather form: no atomics, fixed order)
// Activations between the convs are kept NHWC ([B, OH, OW, C], i.e. the GEMM's natural [M, N]
// output), which makes every im2col read and col2im write contiguous along C; the reference's
// NCHW only matters at the two ends: the uint8 input (read directly, the u8->f32 cast and the
// 1/255 scale of head.py:46 fused into the first im2col) and the flatten feeding `l`
// (jb_nhwc_to_nchw reorders [B,49,64] -> [B,64*49] so the Linear weights keep the reference's
// feature order and checkpoints stay interchangeable).
// K index order of `col` = c*KH*KW + ky*KW + kx = the memory order of torch's conv weight
// [C_out, C_in, KH, KW], so the weight tensor is used as the GEMM's B operand unchanged.
#include "common.cuh"

namespace {

// x: [rows, C, H, W] uint8 (NCHW, the env/replay/rollout layout)  ->  col [B*OH*OW, C*KH*KW] f32, scaled by 1/255.
// Output row b reads input row idx[b] (idx NULL: row b), so a minibatch is gathered inside the im2col.  Row byte
// offsets are 64-bit: a 4x84x84 stack is 28 224 B, so row indices from 76 088 up lie past 2^31 bytes.
__global__ void im2col_u8_nchw_kernel(const uint8_t* __restrict__ x, const int32_t* __restrict__ idx, int B, int C,
                                      int H, int W, int KH, int KW, int S, int OH, int OW, float* __restrict__ col) {
  const int K = C * KH * KW;
  const long long total = (long long)B * OH * OW * K;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(e % K);
    const long long m = e / K;
    const int ox = (int)(m % OW), oy = (int)((m / OW) % OH), b = (int)(m / ((long long)OW * OH));
    const int kx = k % KW, ky = (k / KW) % KH, c = k / (KW * KH);
    const int iy = oy * S + ky, ix = ox * S + kx;
    const long long row = idx ? (long long)idx[b] : (long long)b;
    const float v = (float)x[row * C * H * W + ((size_t)c * H + iy) * W + ix];
    col[e] = v / 255.0f;
  }
}

// Same, four consecutive kx per thread (KW % 4 == 0, S % 4 == 0, W % 4 == 0: the 8x8 stride-4 first layer): one 4-byte
// load of the frame row and one 16-byte store of the column row per thread, 32-bit index arithmetic inside a row.
__global__ void im2col_u8_nchw_vec4_kernel(const uint8_t* __restrict__ x, const int32_t* __restrict__ idx, int B, int C,
                                           int H, int W, int KH, int KW, int S, int OH, int OW, float* __restrict__ col) {
  const int K4 = (C * KH * KW) >> 2, KW4 = KW >> 2;
  const long long total = (long long)B * OH * OW * K4;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int k4 = (int)(e % K4);
    const int m = (int)(e / K4);
    const int ox = m % OW, t = m / OW, oy = t % OH, b = t / OH;
    const int kx4 = k4 % KW4, t2 = k4 / KW4, ky = t2 % KH, c = t2 / KH;
    const long long row = idx ? (long long)idx[b] : (long long)b;
    const uchar4 v = *reinterpret_cast<const uchar4*>(x + row * C * H * W + (c * H + oy * S + ky) * W + ox * S + 4 * kx4);
    reinterpret_cast<float4*>(col)[e] = make_float4((float)v.x / 255.0f, (float)v.y / 255.0f, (float)v.z / 255.0f, (float)v.w / 255.0f);
  }
}

// x: [B, H, W, C] f32 (NHWC)  ->  col [B*OH*OW, C*KH*KW]
__global__ void im2col_nhwc_kernel(const float* __restrict__ x, int B, int C, int H, int W, int KH, int KW, int S,
                                   int OH, int OW, float* __restrict__ col) {
  const int K = C * KH * KW;
  const long long total = (long long)B * OH * OW * K;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(e % K);
    const long long m = e / K;
    const int ox = (int)(m % OW), oy = (int)((m / OW) % OH), b = (int)(m / ((long long)OW * OH));
    const int kx = k % KW, ky = (k / KW) % KH, c = k / (KW * KH);
    col[e] = x[(((size_t)b * H + oy * S + ky) * W + ox * S + kx) * C + c];
  }
}

// dx[b, iy, ix, c] = sum over kernel taps that cover (iy, ix) of dcol[(b, oy, ox), (c, ky, kx)],
// optionally masked by a saved post-ReLU activation act (same NHWC shape).
__global__ void col2im_nhwc_kernel(const float* __restrict__ dcol, int B, int C, int H, int W, int KH, int KW, int S,
                                   int OH, int OW, const float* __restrict__ act, float* __restrict__ dx) {
  const int K = C * KH * KW;
  const long long total = (long long)B * H * W * C;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(e % C);
    const long long p = e / C;
    const int ix = (int)(p % W), iy = (int)((p / W) % H), b = (int)(p / ((long long)W * H));
    float acc = 0.f;
    for (int ky = 0; ky < KH; ++ky) {
      const int ty = iy - ky;
      if (ty < 0 || ty % S) continue;
      const int oy = ty / S;
      if (oy >= OH) continue;
      for (int kx = 0; kx < KW; ++kx) {
        const int tx = ix - kx;
        if (tx < 0 || tx % S) continue;
        const int ox = tx / S;
        if (ox >= OW) continue;
        acc += dcol[(((size_t)b * OH + oy) * OW + ox) * K + (c * KH + ky) * KW + kx];
      }
    }
    if (act) acc = act[e] > 0.f ? acc : 0.f;
    dx[e] = acc;
  }
}

// [B, P, C] <-> [B, C, P]  (P = OH*OW); optional ReLU mask by `act` laid out like the OUTPUT
__global__ void permute_bpc_kernel(const float* __restrict__ x, int B, int P, int C, int to_nchw,
                                   const float* __restrict__ act, float* __restrict__ y) {
  const long long total = (long long)B * P * C;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    // e indexes the OUTPUT
    float v;
    if (to_nchw) {   // y[b, c, p] = x[b, p, c]
      const int p = (int)(e % P), c = (int)((e / P) % C), b = (int)(e / ((long long)P * C));
      v = x[((size_t)b * P + p) * C + c];
    } else {         // y[b, p, c] = x[b, c, p]
      const int c = (int)(e % C), p = (int)((e / C) % P), b = (int)(e / ((long long)P * C));
      v = x[((size_t)b * C + c) * P + p];
    }
    if (act) v = act[e] > 0.f ? v : 0.f;
    y[e] = v;
  }
}

}  // namespace

static int conv_grid(long long total) { return jb_grid_for(total, 256 * 4, 8); }

JB_API int jb_im2col_u8_rows(const uint8_t* x, const int32_t* idx, int B, int C, int H, int W, int KH, int KW, int S,
                             float* col, void* stream) {
  if (!x || !col || B <= 0 || C <= 0 || H < KH || W < KW || S <= 0) return JB_ERR_INVALID;
  const int OH = (H - KH) / S + 1, OW = (W - KW) / S + 1;
  const long long total = (long long)B * OH * OW * C * KH * KW;
  // a gathered row starts where x does modulo 16 only when the row size is a multiple of 16 (4x84x84: 16 x 1 764)
  const bool rows_aligned = !idx || ((long long)C * H * W) % 16 == 0;
  if (KW % 4 == 0 && S % 4 == 0 && W % 4 == 0 && (((uintptr_t)x | (uintptr_t)col) & 15) == 0 && rows_aligned &&
      (long long)B * OH * OW < (1ll << 31))
    im2col_u8_nchw_vec4_kernel<<<conv_grid(total / 4), 256, 0, (cudaStream_t)stream>>>(x, idx, B, C, H, W, KH, KW, S, OH, OW, col);
  else
    im2col_u8_nchw_kernel<<<conv_grid(total), 256, 0, (cudaStream_t)stream>>>(x, idx, B, C, H, W, KH, KW, S, OH, OW, col);
  return jb_check_launch();
}

JB_API int jb_im2col_u8(const uint8_t* x, int B, int C, int H, int W, int KH, int KW, int S, float* col, void* stream) {
  return jb_im2col_u8_rows(x, nullptr, B, C, H, W, KH, KW, S, col, stream);
}

JB_API int jb_im2col_nhwc(const float* x, int B, int C, int H, int W, int KH, int KW, int S, float* col, void* stream) {
  if (!x || !col || B <= 0 || C <= 0 || H < KH || W < KW || S <= 0) return JB_ERR_INVALID;
  const int OH = (H - KH) / S + 1, OW = (W - KW) / S + 1;
  im2col_nhwc_kernel<<<conv_grid((long long)B * OH * OW * C * KH * KW), 256, 0, (cudaStream_t)stream>>>(x, B, C, H, W, KH, KW, S, OH, OW, col);
  return jb_check_launch();
}

JB_API int jb_col2im_nhwc(const float* dcol, int B, int C, int H, int W, int KH, int KW, int S, const float* relu_act,
                          float* dx, void* stream) {
  if (!dcol || !dx || B <= 0 || C <= 0 || H < KH || W < KW || S <= 0) return JB_ERR_INVALID;
  const int OH = (H - KH) / S + 1, OW = (W - KW) / S + 1;
  col2im_nhwc_kernel<<<conv_grid((long long)B * H * W * C), 256, 0, (cudaStream_t)stream>>>(dcol, B, C, H, W, KH, KW, S, OH, OW, relu_act, dx);
  return jb_check_launch();
}

JB_API int jb_nhwc_to_nchw(const float* x, int B, int P, int C, float* y, void* stream) {
  if (!x || !y || B <= 0 || P <= 0 || C <= 0) return JB_ERR_INVALID;
  permute_bpc_kernel<<<conv_grid((long long)B * P * C), 256, 0, (cudaStream_t)stream>>>(x, B, P, C, 1, nullptr, y);
  return jb_check_launch();
}

// y[b,p,c] = x[b,c,p], masked by relu_act (NHWC, may be NULL): gradient of the flatten, fused with
// the ReLU mask of the last conv's output.
JB_API int jb_nchw_to_nhwc(const float* x, int B, int P, int C, const float* relu_act, float* y, void* stream) {
  if (!x || !y || B <= 0 || P <= 0 || C <= 0) return JB_ERR_INVALID;
  permute_bpc_kernel<<<conv_grid((long long)B * P * C), 256, 0, (cudaStream_t)stream>>>(x, B, P, C, 0, relu_act, y);
  return jb_check_launch();
}
