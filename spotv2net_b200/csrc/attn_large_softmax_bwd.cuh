// Softmax + LeakyReLU backward of the large-graph path (attn_large.cu), included there twice: SPOTV2_KERNEL_NAME names the
// kernel and SPOTV2_GA = 1 makes the variant that takes d_alpha [B, H, N(j), N(i)], the gradient through the coefficients
// the forward returned (after dropout), which joins dalpha before the dropout factor.  Two kernels under their own names keep
// the machine code of the one without it exactly what it was.  No include guard: meant to be included more than once.
__global__ void __launch_bounds__(kSmX * kSmY)
SPOTV2_KERNEL_NAME(const float* __restrict__ P_aug, const float* __restrict__ Zraw, float* A,
            float* dA, const float* __restrict__ gii, float* __restrict__ fill, float* dP_aug, int N,
            int H, int HC, int ldp, float slope, const DropoutParams drop
#if SPOTV2_GA
            , const float* __restrict__ d_alpha
#endif
) {
  constexpr bool GA = SPOTV2_GA != 0;
#if !SPOTV2_GA
  const float* const d_alpha = nullptr;
#endif
  extern __shared__ float s_src[];
  __shared__ float red[kSmY][kSmX];
  __shared__ float s_dzii[kSmX];
  const int b = blockIdx.z, h = blockIdx.y, tx = threadIdx.x, ty = threadIdx.y;
  const float* Pb = P_aug + (size_t)b * N * ldp;
  for (int j = ty * kSmX + tx; j < N; j += kSmX * kSmY) s_src[j] = Pb[(size_t)j * ldp + HC + h];
  __syncthreads();
  const int i = blockIdx.x * kSmX + tx;
  const bool live = i < N;
  const int ic = live ? i : N - 1;
  const size_t base = ((size_t)b * H + h) * N * N + ic;
  const float* zc = Zraw ? Zraw + base : nullptr;
  float* ac = A + base;
  float* dc = dA + base;
  const float di = Pb[(size_t)ic * ldp + HC + H + h];
  const float g_ii = gii[((size_t)b * H + h) * N + ic];
  // attention dropout: the forward used alpha * m (m = keep / (1 - p)), so dalpha = m * d(alpha m); A leaves this
  // kernel as alpha * m for the dP product
  const unsigned long long ebase = (((unsigned long long)b * H + h) * N + ic) * N;
  auto mfac = [&](int j) { return drop.p > 0.f ? (dropout_keep(drop, ebase + j) ? drop.scale : 0.f) : 1.f; };
  auto dal = [&](int j) { return GA ? dc[(size_t)j * N] + d_alpha[base + (size_t)j * N] : dc[(size_t)j * N]; };
  float dot = 0.f;
#pragma unroll 8
  for (int j = ty; j < N; j += kSmY) dot = fmaf(ac[(size_t)j * N], dal(j) * mfac(j), dot);
  red[ty][tx] = dot;
  __syncthreads();
  dot = 0.f;
#pragma unroll
  for (int k = 0; k < kSmY; ++k) dot += red[k][tx];
  __syncthreads();
  float dd = 0.f;
#pragma unroll 8
  for (int j = ty; j < N; j += kSmY) {
    const float g = (j == ic) ? g_ii : (zc ? zc[(size_t)j * N] : 0.f);
    const float z = g + s_src[j] + di;
    const float m = mfac(j), al = ac[(size_t)j * N];
    const float dl = al * (dal(j) * m - dot);
    const float dz = z > 0.f ? dl : dl * slope;
    dd += dz;
    if (j == ic) s_dzii[tx] = dz;
    if (live) {
      dc[(size_t)j * N] = dz;
      if (drop.p > 0.f) ac[(size_t)j * N] = al * m;
    }
  }
  red[ty][tx] = dd;
  __syncthreads();
  if (ty == 0 && live) {
    dd = 0.f;
#pragma unroll
    for (int k = 0; k < kSmY; ++k) dd += red[k][tx];
    fill[((size_t)b * H + h) * N + i] = s_dzii[tx] / (float)(N > 1 ? N - 1 : 1);
    dP_aug[((size_t)b * N + i) * ldp + HC + H + h] = dd;
  }
}
