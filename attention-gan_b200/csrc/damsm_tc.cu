// DAMSM word-region similarity on the 5th-generation tensor cores (AGB_MATH_TC_F16 / _BF16).
//
// Replaces the loop body of WordsLoss.get_loss (reference losses/words_loss.py:43-86) and the
// func_attention it calls (networks/attention.py:82-121) with ONE persistent kernel:
//
//   work item  = (image b, word tile c): up to 128 caption words (whole captions, packed by
//                their real lengths, so padded words cost nothing)
//   GEMM1      S[r, n]  = sum_d C_b[d, r] W[n, d]          3 M-tiles of 128 regions, N = 128, K = 256
//   epilogue 1 alpha = softmax over the words of each caption (thread = region: thread-local),
//              e = exp(gamma1 * alpha)  -> 16-bit, written K-major / 128B-swizzled to shared memory
//   GEMM2      V[n, d]  = sum_r e[r, n] C_b[d, r]          M = 128 words, N = 256, K = 320
//   epilogue 2 cos_n = <w_n, V_n> / (|w_n| |V_n|)   (thread = word: thread-local; the region-softmax
//              normaliser cancels in the cosine), m[b, i] = log sum_t exp(gamma2 cos)
//
// Operands reach the tensor core by TMA (128B swizzle, K-major); accumulators live in TMEM:
// columns [0,256) = two S buffers (MMA of M-tile j+1 overlaps epilogue 1 of M-tile j),
// columns [256,512) = V.  Warp roles: 0..11 = three epilogue warpgroups, 12 = TMA producer and
// TMEM allocator, 13 = MMA issuer (448 threads = 14 warps; with 4 warps on an SM sub-partition its 16K registers cap
// every thread at 128).
//
// HBM layout of the pre-packed operands (written by the pack kernels below, 16-bit):
//   Wh [tiles*128, 256]   packed caption words, K-major rows; unused rows are zero
//   Ct [Bi*384, 256]      regions as rows (M operand of GEMM1), rows >= R zero, except that rows 320.. repeat the
//                         regions 256..R-1 of the remainder tile (work sharing between the TMEM lane quarters)
//   Ck [Bi*256, 320]      features as rows (N operand of GEMM2), columns >= R zero
#include <algorithm>
#include <type_traits>

#include "tc_gemm_pairs.cuh"

namespace agb {

int sent_cos_fwd_launch(const float* cnn, const float* rnn, int Bi, int Bc, int D, float eps, float* scos_out,
                        cudaStream_t st);
int damsm_diag_att_maps(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                        const int32_t* cap_lens, int Bi, int T, int D, int R, float gamma1, int row_offset,
                        float* att_out, float* S, float* Bt, cudaStream_t st);
int damsm_pair_att_maps(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                        const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                        int P, int T, int D, int R, float gamma1, float* att_out, cudaStream_t st);
size_t damsm_fp32_workspace_bytes(int Bi, int Bc, int T, int D, int R);
int damsm_fp32_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                   const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1, float gamma2,
                   float eps, const float* dm, const float* gscale, float* dimg, float* dwords, void* workspace,
                   size_t workspace_bytes, cudaStream_t st);

namespace tc {

constexpr int kD = 256;                   // feature dim: K of GEMM1, N of GEMM2
constexpr int kTileN = 128;               // word rows per tile
constexpr int kRRows = 384;               // region rows per image in Ct (3 M-tiles)
constexpr int kRCols = 320;               // region columns per image in Ck / e (5 chunks of 64)
constexpr int kChunk = 128 * 128;         // one [128 x 64] 16-bit K-major tile: 16 KB
// per-item cost model of the pair kernels, in units of one caption word slot (fitted to per-CTA times of the
// streaming backward, scripts/bwd3_timeline.py): fixed part per (word tile, image) item and per caption
constexpr int kItemCost0 = 900, kItemCostCap = 32;
constexpr int kThreads = 448;             // warps 0-11 epilogue, 12 TMA producer (+ TMEM alloc), 13 MMA issuer
constexpr int kSmemW = 0;                 // [4][128 x 64]  resident word tile       64 KB
constexpr int kSmemE = 4 * kChunk;        // [5][128 x 64]  e = exp(gamma1 alpha)    80 KB

template <typename T16> __device__ __forceinline__ T16 cvt16(float v);
template <> __device__ __forceinline__ __half cvt16<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 cvt16<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <typename T16> __device__ __forceinline__ float2 unpack2(uint32_t u);
template <> __device__ __forceinline__ float2 unpack2<__half>(uint32_t u) {
  return __half22float2(*reinterpret_cast<__half2*>(&u));
}
template <> __device__ __forceinline__ float2 unpack2<__nv_bfloat16>(uint32_t u) {
  return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
}

// ---------------------------------------------------------------------------------------------
// pack kernels
// ---------------------------------------------------------------------------------------------
// greedy packing of whole captions into units of <= U word rows (U = 128: one unit per tile; U = 64 in split
// precision: two units per tile, so that no caption straddles a 64-row boundary) and <= U captions.
// tile_cpre[t] = exclusive prefix of the per-item cost estimate of word tile t (see cta_items_balanced).
// unit_first / unit_ncap / nunits (U = 64 only): the caption range of every half tile; nunits = 2 * ntiles
// (a trailing half tile without captions is emitted when the count is odd).
__global__ void tile_pack_kernel(const int32_t* __restrict__ cap_lens, int Bc, int T, int U, int32_t* __restrict__ cap_row,
                                 int32_t* __restrict__ tile_first, int32_t* __restrict__ tile_ncap,
                                 int32_t* __restrict__ ntiles, int32_t* __restrict__ tile_cpre,
                                 int32_t* __restrict__ unit_first, int32_t* __restrict__ unit_ncap,
                                 int32_t* __restrict__ nunits) {
  __shared__ int lens_s[1024];
  const int upt = kTileN / U;                 // units per tile
  int row = 0, unit = 0, first = 0, tfirst = 0;
  int cost = kItemCost0, cpre = 0;
  auto close_unit = [&](int next_first) {
    if (unit_first) {
      unit_first[unit] = first;
      unit_ncap[unit] = next_first - first;
    }
    if ((unit + 1) % upt == 0) {              // the tile is complete
      const int tile = unit / upt;
      tile_first[tile] = tfirst;
      tile_ncap[tile] = next_first - tfirst;
      tile_cpre[tile] = cpre;
      cpre += cost;
      cost = kItemCost0;
      tfirst = next_first;
    }
    ++unit;
    first = next_first;
    row = 0;
  };
  for (int base = 0; base < Bc; base += 1024) {
    const int n = min(1024, Bc - base);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) lens_s[i] = min(max(cap_lens[base + i], 0), T);
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 0; k < n; ++k) {
        const int i = base + k, L = lens_s[k];
        // the epilogues read a caption's TMEM columns in windows of 4: keep the whole window inside the
        // unit (the last accumulator buffer ends at TMEM column 512)
        if (row + ((L + 3) & ~3) > U || i - first == U) close_unit(i);
        cap_row[i] = unit * U + row;
        row += L;
        if (L > 0) cost += ((L + 3) & ~3) + kItemCostCap;
      }
    }
  }
  if (threadIdx.x == 0) {
    close_unit(Bc);
    while (unit % upt != 0) close_unit(Bc);   // pad the last tile with empty units
    const int nt = unit / upt;
    tile_cpre[nt] = cpre;
    ntiles[0] = nt;
    if (nunits) nunits[0] = unit;
  }
}

template <typename T16>
__global__ void pack_words_kernel_tc(const float* __restrict__ words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                                     const int32_t* __restrict__ cap_lens, const int32_t* __restrict__ cap_row,
                                     T16* __restrict__ Wh, T16* __restrict__ Wl, float* __restrict__ pn, int T) {
  const int i = blockIdx.x, t = blockIdx.y;
  const int L = min(max(cap_lens[i], 0), T);
  if (t >= L) return;
  const size_t row = (size_t)cap_row[i] + t;
  const float* src = words + (int64_t)i * ws_b + (int64_t)t * ws_t;
  float ss = 0.f;
  for (int d = threadIdx.x; d < kD; d += blockDim.x) {
    const float v = src[(int64_t)d * ws_d];
    const T16 h = cvt16<T16>(v);
    Wh[row * kD + d] = h;
    if (Wl) Wl[row * kD + d] = cvt16<T16>(v - to_f32(h));       // split precision: w = hi + lo
    ss = fmaf(v, v, ss);
  }
  __shared__ float red[8];
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    pn[row] = sqrtf(tot);
  }
}

// img [Bi,256,R] fp32 -> Ck [Bi*256, 320] (same orientation, padded) and Ct [Bi*384, 256] (transposed)
template <typename T16>
__global__ void pack_img_kernel_tc(const float* __restrict__ img, T16* __restrict__ Ck, T16* __restrict__ Ct,
                                   T16* __restrict__ Ckl, T16* __restrict__ Ctl, int R) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, d0 = blockIdx.y * 32, r0 = blockIdx.x * 32;  // r0 < 384
  const int tx = threadIdx.x, ty = threadIdx.y;                            // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int d = d0 + k, r = r0 + tx;
    const float v = (r < R) ? img[((size_t)b * kD + d) * R + r] : 0.f;
    tile[k][tx] = v;
    if (r < kRCols) {
      const T16 h = cvt16<T16>(v);
      Ck[((size_t)b * kD + d) * kRCols + r] = h;
      if (Ckl) Ckl[((size_t)b * kD + d) * kRCols + r] = cvt16<T16>(v - to_f32(h));
    }
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int r = r0 + k, d = d0 + tx;
    const float v = tile[tx][k];
    const T16 h = cvt16<T16>(v);
    const T16 l = cvt16<T16>(v - to_f32(h));
    const bool dup_target = r >= 320 && r - 64 < R;       // written below by the block that owns region r - 64
    if (!dup_target) {
      Ct[((size_t)b * kRRows + r) * kD + d] = h;
      if (Ctl) Ctl[((size_t)b * kRRows + r) * kD + d] = l;
    }
    // the regions of the third (remainder) tile once more in its lanes 64..127 (rows 320..): the pair kernels let
    // lane quarters 2, 3 work on them with the other half of the captions (see `dup` in the epilogues)
    if (r >= 256 && r < R && r + 64 < kRRows) {
      Ct[((size_t)b * kRRows + r + 64) * kD + d] = h;
      if (Ctl) Ctl[((size_t)b * kRRows + r + 64) * kD + d] = l;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// candidate packing (agb_damsm_cand_fwd, agb_damsm_pairs_fwd): every image owns a range of entries (virtual
// captions), [b*K, (b+1)*K) for K candidates per image or CSR offsets eoff[b] .. eoff[b+1] for a pair list grouped
// by image.  The entries are packed by the rule of tile_pack_kernel into units of U rows (U = 64 in split
// precision) that never mix two images.  An image's range is cut into segments of S entries counted from its first
// entry (S = 64 units of the widest captions, see make_plan), and every segment is padded to whole tiles.  An item
// of the pair kernels is one unit.  An entry whose caption index is outside [0, Bc) becomes an entry of length 0,
// whose m the pair kernel writes as NaN.
// ---------------------------------------------------------------------------------------------
// upper bound of one item's cost (kItemCost0 + per live caption its window and kItemCostCap, at most 128 captions
// and 128 + 3 * 128 window rows): the host bounds the cost prefix of a call with it
constexpr int kMaxItemCost = kItemCost0 + kTileN * (kItemCostCap + 4);

__device__ __forceinline__ int ent_off(const int32_t* eoff, int K, int b) { return eoff ? eoff[b] : b * K; }

// the image whose (non-empty) entry range holds entry g < number of entries
__device__ __forceinline__ int ent_img(const int32_t* eoff, int K, int Bi, int g) {
  if (!eoff) return g / K;
  int lo = 0, hi = Bi - 1;                     // the last b with eoff[b] <= g
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (eoff[mid] <= g) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// One warp per window of S consecutive entries: it packs, in image order, every segment that starts inside the
// window, in lock-step (lane k % 32 loads entry k of the segment).  A segment holds at most S entries, so no warp
// walks more than 2 S entries however skewed the ranges are.  Pass 1 (!kWrite): the window's item count and cost
// into win_items / win_cost.  Pass 2 (kWrite, after cand_scan_kernel turned them into exclusive prefixes): cap_row,
// vlen of every entry, first entry / entry count / cost prefix of every item, image of every tile.  With K <= S
// every image is one segment, and the layout is that of one warp per image.
template <bool kWrite>
__global__ void __launch_bounds__(256)
cand_pack_kernel(const int32_t* __restrict__ cap_lens, int Bc, int T, const int32_t* __restrict__ cand,
                 const int32_t* __restrict__ eoff, int Bi, int K, int nwin, int S, int U,
                 int32_t* __restrict__ win_items, int32_t* __restrict__ win_cost, int32_t* __restrict__ cap_row,
                 int32_t* __restrict__ vlen, int32_t* __restrict__ item_first, int32_t* __restrict__ item_ncap,
                 int32_t* __restrict__ cpre, int32_t* __restrict__ tile_img) {
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= nwin) return;
  const int nent = ent_off(eoff, K, Bi);
  const long long g0 = (long long)w * S, g1 = min((long long)nent, g0 + S);
  const int upt = kTileN / U;
  const int item0 = kWrite ? win_items[w] : 0, cost0 = kWrite ? win_cost[w] : 0;
  int unit = 0, cacc = 0;
  for (long long g = g0; g < g1;) {
    const int b = ent_img(eoff, K, Bi, (int)g);
    const int e0 = ent_off(eoff, K, b), e1 = ent_off(eoff, K, b + 1);
    const long long s0 = e0 + (g - e0 + S - 1) / S * S;   // image b's first segment start at or after g
    g = e1;
    if (s0 >= g1 || s0 >= e1) continue;          // no segment of image b starts in this window
    const int v0 = (int)s0, cnt = (int)(min((long long)e1, s0 + S) - s0);
    int row = 0, first = 0, cost = kItemCost0;
    auto close_unit = [&](int next_first) {
      if (kWrite && lane == 0) {
        const int it = item0 + unit;
        item_first[it] = v0 + first;
        item_ncap[it] = next_first - first;
        cpre[it] = cost0 + cacc;
        if (it % upt == 0) tile_img[it / upt] = b;
      }
      cacc += cost;
      cost = kItemCost0;
      ++unit;
      first = next_first;
      row = 0;
    };
    for (int k0 = 0; k0 < cnt; k0 += 32) {
      int myL = 0;
      if (k0 + lane < cnt) {
        const int j = cand[(size_t)v0 + k0 + lane];
        myL = (j >= 0 && j < Bc) ? min(max(cap_lens[j], 0), T) : 0;
      }
      const int n = min(32, cnt - k0);
      for (int i = 0; i < n; ++i) {
        const int k = k0 + i, L = __shfl_sync(0xffffffffu, myL, i);
        if (row + ((L + 3) & ~3) > U || k - first == U) close_unit(k);
        if (kWrite && lane == i) {
          cap_row[v0 + k] = (item0 + unit) * U + row;
          vlen[v0 + k] = L;
        }
        row += L;
        if (L > 0) cost += ((L + 3) & ~3) + kItemCostCap;
      }
    }
    close_unit(cnt);
    while (unit % upt != 0) close_unit(cnt);   // pad the segment to whole tiles with empty units
  }
  if (!kWrite && lane == 0) {
    win_items[w] = unit;
    win_cost[w] = cacc;
  }
}

// exclusive prefix over the windows of their item counts and costs (one block); the totals give the number of
// tiles / units and the end of the cost prefix
__global__ void __launch_bounds__(1024)
cand_scan_kernel(int32_t* __restrict__ win_items, int32_t* __restrict__ win_cost, int n, int upt,
                 int32_t* __restrict__ cpre, int32_t* __restrict__ ntiles, int32_t* __restrict__ nunits) {
  __shared__ int si[1024], sc[1024];
  const int tid = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int lo = min(n, tid * per), hi = min(n, lo + per);
  int a = 0, c = 0;
  for (int b = lo; b < hi; ++b) {
    a += win_items[b];
    c += win_cost[b];
  }
  si[tid] = a;
  sc[tid] = c;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int pa = tid >= o ? si[tid - o] : 0, pc = tid >= o ? sc[tid - o] : 0;
    __syncthreads();
    si[tid] += pa;
    sc[tid] += pc;
    __syncthreads();
  }
  int ra = si[tid] - a, rc = sc[tid] - c;
  for (int b = lo; b < hi; ++b) {
    const int x = win_items[b], y = win_cost[b];
    win_items[b] = ra;
    win_cost[b] = rc;
    ra += x;
    rc += y;
  }
  if (tid == 1023) {
    cpre[si[tid]] = sc[tid];
    ntiles[0] = si[tid] / upt;
    if (nunits) nunits[0] = si[tid];
  }
}

// One block per word tile: the 16-bit rows (hi, and lo in split precision) and norms of the tile's virtual
// captions, straight from the caller's fp32 words; rows no caption uses are zero.  The arithmetic (conversion,
// the norm's summation order) is that of pack_words_kernel_tc, so a candidate pair sees the same operands as the
// same pair in agb_damsm_fwd.
template <typename T16>
__global__ void __launch_bounds__(512)
cand_rows_kernel(const float* __restrict__ words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                 const int32_t* __restrict__ cand, const int32_t* __restrict__ vlen, const int32_t* __restrict__ cap_row,
                 const int32_t* __restrict__ item_first, const int32_t* __restrict__ item_ncap, int U,
                 const int32_t* __restrict__ ntiles, T16* __restrict__ Wh, T16* __restrict__ Wl, float* __restrict__ pn) {
  __shared__ int src_j[kTileN];
  __shared__ unsigned char src_t[kTileN];
  __shared__ float red[kTileN][4];
  const int tile = blockIdx.x;
  if (tile >= ntiles[0]) return;
  if (threadIdx.x < kTileN) src_j[threadIdx.x] = -1;
  __syncthreads();
  const int upt = kTileN / U;
  for (int s = 0; s < upt; ++s) {
    const int first = item_first[tile * upt + s], n = item_ncap[tile * upt + s];
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const int v = first + e, L = vlen[v];
      const int r0 = cap_row[v] - tile * kTileN, j = cand[v];
      for (int t = 0; t < L; ++t) {
        src_j[r0 + t] = j;
        src_t[r0 + t] = (unsigned char)t;
      }
    }
  }
  __syncthreads();
  const int x = threadIdx.x & 127, g = threadIdx.x >> 7;
#pragma unroll 4
  for (int r = g; r < kTileN; r += 4) {
    const int j = src_j[r];
    float v0 = 0.f, v1 = 0.f;
    if (j >= 0) {
      const float* src = words + (int64_t)j * ws_b + (int64_t)src_t[r] * ws_t;
      v0 = src[(int64_t)x * ws_d];
      v1 = src[(int64_t)(x + 128) * ws_d];
    }
    const size_t row = (size_t)tile * kTileN + r;
    const T16 h0 = cvt16<T16>(v0), h1 = cvt16<T16>(v1);
    Wh[row * kD + x] = h0;
    Wh[row * kD + x + 128] = h1;
    if (Wl) {
      Wl[row * kD + x] = cvt16<T16>(v0 - to_f32(h0));
      Wl[row * kD + x + 128] = cvt16<T16>(v1 - to_f32(h1));
    }
    float ss = fmaf(v0, v0, 0.f);
    ss = fmaf(v1, v1, ss);
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[r][x >> 5] = ss;
  }
  __syncthreads();
  if (threadIdx.x < kTileN) {
    float tot = 0.f;
    for (int w = 0; w < 4; ++w) tot += red[threadIdx.x][w];
    pn[(size_t)tile * kTileN + threadIdx.x] = sqrtf(tot);
  }
}

// ---------------------------------------------------------------------------------------------
// pair lists (agb_damsm_pairs_fwd): the pairs are grouped by image with a stable counting sort on the image index,
// as a least-significant-digit radix sort over two 8-bit digits.  Each pass is a per-block digit histogram, one
// exclusive scan over (digit, block), and a stable scatter.  A pair whose image is outside [0, Bi) gets key 0xffff
// (Bi <= 65535 keeps it free), which sorts after every image and is not packed.  Integer counts only: the order is
// deterministic, and inside an image the pairs keep their list order.
// ---------------------------------------------------------------------------------------------
constexpr int kSortTile = 2048;                // pairs per block of a sort pass (8 per thread)

__device__ __forceinline__ int pair_key(const int32_t* __restrict__ pair_img, int Bi, long long p) {
  const int b = pair_img[p];
  return (b >= 0 && b < Bi) ? b : 0xffff;
}

// digit counts of one block's pairs: hist[digit * gridDim.x + block].  kin == nullptr: keys from pair_img
__global__ void __launch_bounds__(256)
pair_hist_kernel(const int32_t* __restrict__ pair_img, int Bi, const int32_t* __restrict__ kin, long long P, int shift,
                 int32_t* __restrict__ hist) {
  __shared__ int cnt[256];
  cnt[threadIdx.x] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < kSortTile; i += 256) {
    const long long p = (long long)blockIdx.x * kSortTile + i;
    if (p < P) atomicAdd(&cnt[((kin ? kin[p] : pair_key(pair_img, Bi, p)) >> shift) & 255], 1);
  }
  __syncthreads();
  hist[threadIdx.x * gridDim.x + blockIdx.x] = cnt[threadIdx.x];
}

// in-place exclusive prefix of n ints (one block)
__global__ void __launch_bounds__(1024) excl_scan_kernel(int32_t* __restrict__ a, int n) {
  __shared__ int s[1024];
  const int tid = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int lo = min(n, tid * per), hi = min(n, lo + per);
  int acc = 0;
  for (int i = lo; i < hi; ++i) acc += a[i];
  s[tid] = acc;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int pv = tid >= o ? s[tid - o] : 0;
    __syncthreads();
    s[tid] += pv;
    __syncthreads();
  }
  int r = s[tid] - acc;
  for (int i = lo; i < hi; ++i) {
    const int x = a[i];
    a[i] = r;
    r += x;
  }
}

// stable scatter of one block's pairs to their digit's slots: rounds of 256 pairs in list order; inside a round the
// rank of a pair is its lane rank among the warp's pairs of the same digit plus the counts of the earlier warps.
// kin == nullptr: keys from pair_img, values = pair indices
__global__ void __launch_bounds__(256)
pair_scatter_kernel(const int32_t* __restrict__ pair_img, int Bi, const int32_t* __restrict__ kin,
                    const int32_t* __restrict__ vin, long long P, int shift, const int32_t* __restrict__ hist,
                    int32_t* __restrict__ kout, int32_t* __restrict__ vout) {
  __shared__ int base[256];
  __shared__ int wcnt[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  base[threadIdx.x] = hist[threadIdx.x * gridDim.x + blockIdx.x];
  for (int w = 0; w < 8; ++w) wcnt[w][threadIdx.x] = 0;
  __syncthreads();
  for (int r0 = 0; r0 < kSortTile; r0 += 256) {
    const long long p = (long long)blockIdx.x * kSortTile + r0 + threadIdx.x;
    const bool live = p < P;
    int key = 0, val = 0, d = 256;
    if (live) {
      key = kin ? kin[p] : pair_key(pair_img, Bi, p);
      val = kin ? vin[p] : (int)p;
      d = (key >> shift) & 255;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (live && rank == 0) wcnt[warp][d] = __popc(peers);
    __syncthreads();
    if (live) {
      int pos = base[d] + rank;
      for (int w = 0; w < warp; ++w) pos += wcnt[w][d];
      kout[pos] = key;
      vout[pos] = val;
    }
    __syncthreads();
    int tot = 0;
    for (int w = 0; w < 8; ++w) {
      tot += wcnt[w][threadIdx.x];
      wcnt[w][threadIdx.x] = 0;
    }
    base[threadIdx.x] += tot;
    __syncthreads();
  }
}

// thread t <= Bi: eoff[t] = the first sorted pair of image t (eoff[Bi] = number of pairs with a valid image);
// thread t < P: the caption index of sorted pair t
__global__ void __launch_bounds__(256)
pair_offsets_kernel(const int32_t* __restrict__ key, const int32_t* __restrict__ val,
                    const int32_t* __restrict__ pair_cap, int P, int Bi, int32_t* __restrict__ eoff,
                    int32_t* __restrict__ cap_sorted) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t <= Bi) {
    int lo = 0, hi = P;                        // the first sorted position with key >= t
    while (lo < hi) {
      const int mid = (int)(((long long)lo + hi) >> 1);
      if (key[mid] < t) lo = mid + 1;
      else hi = mid;
    }
    eoff[t] = lo;
  }
  if (t < P) cap_sorted[t] = pair_cap[val[t]];
}

// m from packed (sorted) order back to list order; pairs with an invalid image get NaN
__global__ void __launch_bounds__(256)
pair_scatter_m_kernel(const float* __restrict__ m_sorted, const int32_t* __restrict__ val,
                      const int32_t* __restrict__ eoff, int Bi, int P, float* __restrict__ m_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  m_out[val[i]] = i < eoff[Bi] ? m_sorted[i] : __int_as_float(0x7fc00000);
}

// ---------------------------------------------------------------------------------------------
// epilogue 1 for one caption and one region (thread): NL = caption length rounded up to 4.
// Branch-free: slots t >= L are set to -inf (their exponentials are 0) and only their stores are
// predicated; slots below NL-4 are always live, so they carry no predicate at all.
// ---------------------------------------------------------------------------------------------
template <typename T16> __device__ __forceinline__ uint16_t bits16(float v) {
  const T16 h = cvt16<T16>(v);
  return *reinterpret_cast<const uint16_t*>(&h);
}

// K region tiles at once (K = 2: the two score buffers of region tiles 0 and 1 are processed together,
// which gives every thread two independent dependency chains to overlap MUFU / TMEM latencies)
template <typename T16, int NL, int K>
__device__ __forceinline__ void caption_softmax(const uint32_t (&taddr)[K], int L, int off, const int (&r)[K], int R,
                                                uint32_t sE32, float scale_log2, float g1_log2) {
  float s[K][NL];
#pragma unroll
  for (int k = 0; k < K; ++k) tmem_ld_n<NL>(taddr[k], s[k]);
  tmem_ld_wait();
  uint32_t colbase[K], x[K];
  bool store[K], live[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    // element (row n, col r) of the K-major 128B-swizzled e tile: chunk (r>>6), 16-byte unit ((r&63)>>3) ^ (n&7)
    colbase[k] = sE32 + (uint32_t)(r[k] >> 6) * kChunk + ((r[k] & 7) << 1) + (uint32_t)off * 128;
    x[k] = ((r[k] & 63) >> 3) << 4;
    store[k] = r[k] < kRCols;
    live[k] = r[k] < R;          // padding regions (R <= r < 320) contribute zeros to V
  }
  float ksc[K], mxs[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int t = NL - 4; t < NL; ++t)
      if (t >= L) s[k][t] = -INFINITY;
    float m4[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) m4[i] = s[k][i];
#pragma unroll
    for (int t = 4; t < NL; ++t) m4[t & 3] = fmaxf(m4[t & 3], s[k][t]);
    mxs[k] = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * scale_log2;
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int t = 0; t < NL; ++t) {
      s[k][t] = exp2f(fmaf(s[k][t], scale_log2, -mxs[k]));  // exp((s - max)/sqrt(D))
      s4[t & 3] += s[k][t];
    }
    ksc[k] = g1_log2 / ((s4[0] + s4[1]) + (s4[2] + s4[3]));
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int t = 0; t < NL; ++t) {
      const uint16_t e = live[k] ? bits16<T16>(exp2f(s[k][t] * ksc[k])) : (uint16_t)0;  // exp(gamma1 alpha)
      if (store[k] && (t < NL - 4 || t < L)) st_shared_u16(colbase[k] + t * 128 + ((((off + t) << 4) & 0x70) ^ x[k]), e);
    }
  }
}

#define AGB_CAPTION_SWITCH(L, CALL)                       \
  switch (((L) + 3) >> 2) {                               \
    case 1: { constexpr int NL = 4; CALL; } break;        \
    case 2: { constexpr int NL = 8; CALL; } break;        \
    case 3: { constexpr int NL = 12; CALL; } break;       \
    case 4: { constexpr int NL = 16; CALL; } break;       \
    case 5: { constexpr int NL = 20; CALL; } break;       \
    case 6: { constexpr int NL = 24; CALL; } break;       \
    case 7: { constexpr int NL = 28; CALL; } break;       \
    default: { constexpr int NL = 32; CALL; } break;      \
  }

struct FwdParams {
  const int32_t* tile_first;
  const int32_t* tile_ncap;
  const int32_t* ntiles;
  const int32_t* cap_row;
  const int32_t* cap_lens;
  const int32_t* tile_cpre;   // [ntiles + 1] exclusive prefix of the per-item cost of each word tile
  int uniform_split;          // != 0: equal item counts per CTA instead of equal cost (option damsm_uniform_split, for A/B timing)
  int dup_rem;                // != 0: region tile 2 carries its regions twice (lanes 0..63 and 64..127, see pack_img_kernel_tc)
  int img_block;              // > 0: item order (image block, word tile, image) with this many images per block (item_pos)
  const float* pn;
  float* m_out;
  int Bi, Bc, T, R;
  float scale_log2, g1_log2, gamma2;
  // training forward (kSave) / streaming backward: saved per (image, word row), Ntot = nt_max * 128 rows per image
  void* v16;             // [Bi, Ntot, 256] 16-bit normalised context vectors
  float4* rowst;         // [Bi, Ntot] {<w,v>, |v|, 1/Z, -}
  int Ntot;
};

// candidate mode (agb_damsm_cand_fwd): the captions are virtual (entry v = b*K + k is a copy of caption cand[b,k]),
// every word tile belongs to one image, and a work item is one word tile.  tile_first / tile_ncap / cap_row /
// cap_lens / tile_cpre describe the virtual captions, m_out is [Bi*K] indexed by v.
struct FwdCandParams : FwdParams {
  const int32_t* tile_img;   // [ntiles] image of every word tile
  const void* wh;            // packed words (Wh): epilogue 2 reads <w, V> from here, not from the resident tile
};

// tile_img of candidate mode; the dense kernels never read it
__device__ __forceinline__ const int32_t* cand_tile_img(const FwdParams&) { return nullptr; }
__device__ __forceinline__ const int32_t* cand_tile_img(const FwdCandParams& p) { return p.tile_img; }

#include "damsm_tc_fwd2.inc"
#include "damsm_tc_fwd2x.inc"

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct TcPlan {
  int nt_max;
  size_t off_Wh, off_pn, off_caprow, off_tfirst, off_tncap, off_tcpre, off_ntiles, off_Ct, off_Ck, off_attS, off_attB;
  // fused backward staging, per chunk of ct word tiles (N = ct*128 word rows) and all Bi images
  int ct;        // tiles per chunk
  int splits;    // slices of the image range in the d words GEMM
  size_t off_E16, off_dV16, off_A116, off_dpp, off_dwp, off_m, total;
  // what the training forward saves for the streaming backward (damsm_bwd3_kernel); save == 0: the saved
  // context vectors would not fit the budget (or AGB_DAMSM_BWD=2) and the backward recomputes (damsm_bwd2_kernel)
  int save;
  size_t off_v16, off_rowst;
  // split precision (AGB_MATH_TC_F16X2): captions packed into 64-row half tiles, lo parts of every operand
  int split;
  size_t off_Wl, off_Ctl, off_Ckl, off_ufirst, off_uncap, off_nunits;
};

static TcPlan make_tc_plan(int Bi, int Bc, int T, int D, int R, bool split) {
  const Options& opt = options();
  TcPlan p;
  p.split = split ? 1 : 0;
  const int window = (T + 3) & ~3;              // a caption's TMEM columns are read in windows of 4
  if (split) {
    const int per_unit = 64 / window;           // captions that always fit in one 64-row half tile
    p.nt_max = ((Bc + per_unit - 1) / per_unit + 1) / 2;
  } else {
    const int per_tile = 128 / window;          // captions that always fit in one tile
    p.nt_max = (Bc + per_tile - 1) / per_tile;
  }
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 1024); return at; };
  p.off_Wh = take((size_t)p.nt_max * kTileN * kD * 2);
  p.off_pn = take((size_t)p.nt_max * kTileN * 4);
  p.off_caprow = take((size_t)Bc * 4);
  p.off_tfirst = take((size_t)p.nt_max * 4);
  p.off_tncap = take((size_t)p.nt_max * 4);
  p.off_tcpre = take((size_t)(p.nt_max + 1) * 4);
  p.off_ntiles = take(256);
  p.off_Ct = take((size_t)Bi * kRRows * kD * 2);
  p.off_Ck = take((size_t)Bi * kD * kRCols * 2);
  p.off_attS = take((size_t)Bi * T * R * 4);
  p.off_attB = take((size_t)Bi * T * R * 4);
  p.off_Wl = p.off_Ctl = p.off_Ckl = p.off_ufirst = p.off_uncap = p.off_nunits = 0;
  if (split) {
    p.off_Wl = take((size_t)p.nt_max * kTileN * kD * 2);
    p.off_Ctl = take((size_t)Bi * kRRows * kD * 2);
    p.off_Ckl = take((size_t)Bi * kD * kRCols * 2);
    p.off_ufirst = take((size_t)2 * p.nt_max * 4);
    p.off_uncap = take((size_t)2 * p.nt_max * 4);
    p.off_nunits = take(256);
  }
  const size_t all_rows = (size_t)Bi * p.nt_max * kTileN;
  p.save = (all_rows * (kD * 2 + 16) <= (size_t)std::max<long long>(0, opt.damsm_save_bytes) && opt.damsm_bwd != 2) ? 1 : 0;
  // staging of one backward chunk: E16 + A116 (+ dV16 for the recomputing backward) + dpp per (image, word row)
  const size_t tile_bytes = (size_t)Bi * kTileN * (kRCols * 2 * 2 + (p.save ? 0 : kD * 2) + 4);
  size_t ct = (size_t)std::max<long long>(0, opt.damsm_chunk_bytes) / tile_bytes;
  if (ct < 1) ct = 1;
  if (ct > (size_t)p.nt_max) ct = p.nt_max;
  p.ct = (int)ct;
  p.splits = std::max(1, std::min(Bi, opt.damsm_dw_splits));
  const size_t rows = (size_t)Bi * ct * kTileN;
  p.off_E16 = take(rows * kRCols * 2);
  p.off_dV16 = p.save ? p.off_E16 : take(rows * kD * 2);
  p.off_A116 = take(rows * kRCols * 2);
  p.off_dpp = take(rows * 4);
  p.off_dwp = take((size_t)p.splits * ct * kTileN * kD * 4);
  p.off_m = take((size_t)Bi * Bc * 4);
  p.off_v16 = p.off_rowst = o;
  if (p.save) {
    p.off_v16 = take(all_rows * kD * 2);
    p.off_rowst = take(all_rows * 16);
  }
  p.total = o;
  return p;
}

static int num_sms() { return device_sms(); }

struct Packed {
  void* Wh; float* pn; int32_t *cap_row, *tfirst, *tncap, *tcpre, *ntiles; void* Ct; void* Ck;
  void *Wl, *Ctl, *Ckl; int32_t *ufirst, *uncap, *nunits;     // split precision only
};

// pack the operands of one call: caption tiles, 16-bit words, 16-bit region features (both layouts)
template <typename T16>
static int run_pack(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                    const int32_t* cap_lens, int Bi, int Bc, int T, int R, char* ws, const TcPlan& pl, Packed* out,
                    cudaStream_t st, bool already_packed = false) {
  T16* Wh = (T16*)(ws + pl.off_Wh);
  float* pn = (float*)(ws + pl.off_pn);
  int32_t* cap_row = (int32_t*)(ws + pl.off_caprow);
  int32_t* tfirst = (int32_t*)(ws + pl.off_tfirst);
  int32_t* tncap = (int32_t*)(ws + pl.off_tncap);
  int32_t* tcpre = (int32_t*)(ws + pl.off_tcpre);
  int32_t* ntiles = (int32_t*)(ws + pl.off_ntiles);
  T16* Ct = (T16*)(ws + pl.off_Ct);
  T16* Ck = (T16*)(ws + pl.off_Ck);
  T16* Wl = pl.split ? (T16*)(ws + pl.off_Wl) : nullptr;
  T16* Ctl = pl.split ? (T16*)(ws + pl.off_Ctl) : nullptr;
  T16* Ckl = pl.split ? (T16*)(ws + pl.off_Ckl) : nullptr;
  int32_t* ufirst = pl.split ? (int32_t*)(ws + pl.off_ufirst) : nullptr;
  int32_t* uncap = pl.split ? (int32_t*)(ws + pl.off_uncap) : nullptr;
  int32_t* nunits = pl.split ? (int32_t*)(ws + pl.off_nunits) : nullptr;
  if (!already_packed) {
    // Wh and pn are neighbours in the workspace: one memset for both (unused word rows must read as zero)
    AGB_CUDA(cudaMemsetAsync(Wh, 0, (pl.off_pn - pl.off_Wh) + (size_t)pl.nt_max * kTileN * 4, st));
    if (Wl) AGB_CUDA(cudaMemsetAsync(Wl, 0, (size_t)pl.nt_max * kTileN * kD * 2, st));
    tile_pack_kernel<<<1, 256, 0, st>>>(cap_lens, Bc, T, pl.split ? 64 : kTileN, cap_row, tfirst, tncap, ntiles, tcpre,
                                        ufirst, uncap, nunits);
    if (int rc = check_launch("tile_pack_kernel")) return rc;
    pack_words_kernel_tc<T16><<<dim3(Bc, T), 128, 0, st>>>(words, ws_b, ws_d, ws_t, cap_lens, cap_row, Wh, Wl, pn, T);
    if (int rc = check_launch("pack_words_kernel_tc")) return rc;
    pack_img_kernel_tc<T16><<<dim3(kRRows / 32, kD / 32, Bi), dim3(32, 8), 0, st>>>(img, Ck, Ct, Ckl, Ctl, R);
    if (int rc = check_launch("pack_img_kernel_tc")) return rc;
  }
  out->Wl = Wl; out->Ctl = Ctl; out->Ckl = Ckl; out->ufirst = ufirst; out->uncap = uncap; out->nunits = nunits;
  out->Wh = Wh; out->pn = pn; out->cap_row = cap_row; out->tfirst = tfirst; out->tncap = tncap; out->tcpre = tcpre; out->ntiles = ntiles;
  out->Ct = Ct; out->Ck = Ck;
  return 0;
}

template <typename T16>
static int launch_fwd(const Packed& pk, const int32_t* cap_lens, int Bi, int Bc, int T, int R, float gamma1,
                      float gamma2, float* m_out, char* ws, const TcPlan& pl, bool save, cudaStream_t st);

template <typename T16>
static int run_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                   const int32_t* cap_lens, int Bi, int Bc, int T, int R, float gamma1, float gamma2, float* m_out,
                   char* ws, const TcPlan& pl, bool save, cudaStream_t st) {
  Packed pk;
  if (int rc = run_pack<T16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, R, ws, pl, &pk, st)) return rc;
  return launch_fwd<T16>(pk, cap_lens, Bi, Bc, T, R, gamma1, gamma2, m_out, ws, pl, save, st);
}

template <typename T16>
static int launch_fwd(const Packed& pk, const int32_t* cap_lens, int Bi, int Bc, int T, int R, float gamma1,
                      float gamma2, float* m_out, char* ws, const TcPlan& pl, bool save, cudaStream_t st) {
  save = save && pl.save;
  const bool bf = std::is_same<T16, __nv_bfloat16>::value;
  CUtensorMap mapW, mapCt, mapCk;
  if (int rc = make_tmap_2d(&mapW, pk.Wh, (uint64_t)pl.nt_max * kTileN, kD, 128, bf)) return rc;
  if (int rc = make_tmap_2d(&mapCt, pk.Ct, (uint64_t)Bi * kRRows, kD, 128, bf)) return rc;
  if (int rc = make_tmap_2d(&mapCk, pk.Ck, (uint64_t)Bi * kD, kRCols, 128, bf)) return rc;
  FwdParams p;
  p.tile_first = pk.tfirst; p.tile_ncap = pk.tncap; p.ntiles = pk.ntiles; p.cap_row = pk.cap_row; p.cap_lens = cap_lens;
  p.tile_cpre = pk.tcpre;
  p.uniform_split = options().damsm_uniform_split;
  p.img_block = options().damsm_img_block;
  p.dup_rem = R > 256 ? 1 : 0;
  p.pn = pk.pn; p.m_out = m_out; p.Bi = Bi; p.Bc = Bc; p.T = T; p.R = R;
  p.scale_log2 = kLog2e / sqrtf((float)kD);
  p.g1_log2 = gamma1 * kLog2e;
  p.gamma2 = gamma2;
  p.v16 = ws + pl.off_v16; p.rowst = (float4*)(ws + pl.off_rowst); p.Ntot = pl.nt_max * kTileN;
  if (pl.split) {
    if constexpr (std::is_same<T16, __half>::value) {
      CUtensorMap mapWh, mapWl, mapCtl, mapCkl;
      if (int rc = make_tmap_2d(&mapWh, pk.Wh, (uint64_t)pl.nt_max * kTileN, kD, 64, false)) return rc;
      if (int rc = make_tmap_2d(&mapWl, pk.Wl, (uint64_t)pl.nt_max * kTileN, kD, 64, false)) return rc;
      if (int rc = make_tmap_2d(&mapCtl, pk.Ctl, (uint64_t)Bi * kRRows, kD, 128, false)) return rc;
      if (int rc = make_tmap_2d(&mapCkl, pk.Ckl, (uint64_t)Bi * kD, kRCols, 128, false)) return rc;
      FwdXParams xp;
      xp.f = p; xp.unit_first = pk.ufirst; xp.unit_ncap = pk.uncap; xp.nunits = pk.nunits;
      auto kx = save ? damsm_fwd2x_kernel<true> : damsm_fwd2x_kernel<false>;
      AGB_CUDA(cudaFuncSetAttribute(kx, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes2));
      const long long max_items_x = (long long)Bi * pl.nt_max * 2;
      const int grid_x = (int)std::min<long long>(num_sms(), max_items_x);
      const int slot_x = prof_begin(PROF_DAMSM_TC_FWD, st);
      kx<<<grid_x, kThreads, kSmemBytes2, st>>>(mapWh, mapWl, mapCt, mapCtl, mapCk, mapCkl, xp);
      prof_end(slot_x, st);
      return check_launch("damsm_fwd2x_kernel");
    } else {
      return fail_unsupported("split precision needs fp16 operands");
    }
  }
  auto kern = save ? damsm_fwd2_kernel<T16, true> : damsm_fwd2_kernel<T16, false>;
  AGB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes2));
  const long long max_items = (long long)Bi * pl.nt_max;
  const int grid = (int)std::min<long long>(num_sms(), max_items);
  const int slot = prof_begin(PROF_DAMSM_TC_FWD, st);
  kern<<<grid, kThreads, kSmemBytes2, st>>>(mapW, mapCt, mapCk, p);
  prof_end(slot, st);
  return check_launch("damsm_fwd_kernel");
}

// ---------------------------------------------------------------------------------------------
// candidate mode: workspace plan from shapes only (the caption lengths stay on the device)
// ---------------------------------------------------------------------------------------------
struct CandPlan {
  int split, S;                  // S: entries per packing segment (see cand_pack_kernel)
  long long nent, nwin, items_max, nt_max, sort_blocks;   // items: word tiles, or 64-row units in split precision
  size_t off_Wh, off_Wl, off_pn, off_caprow, off_vlen, off_ifirst, off_incap, off_cpre, off_timg, off_iitems, off_icost,
      off_counts, off_Ct, off_Ck, off_Ctl, off_Ckl, total;
  // pair lists only: sort buffers (keys, values: pass 1 -> A, pass 2 -> B), digit histogram, CSR offsets, the
  // caption index of every sorted pair and m in sorted order
  size_t off_keyA, off_valA, off_keyB, off_valB, off_hist, off_eoff, off_capS, off_mS;
};

// nent entries over Bi images, at most items_max items (units).  S = 64 units of the widest captions: an even
// number of units, so that cutting a range into segments never needs more units than packing it whole (every
// closed unit holds at least per_unit captions).
static CandPlan make_plan(int Bi, long long nent, long long items_max, int T, bool split, bool pairs) {
  CandPlan p;
  p.split = split ? 1 : 0;
  const int U = split ? 64 : kTileN;
  const int window = (T + 3) & ~3;
  p.S = 64 * (U / window);
  p.nent = nent;
  p.nwin = (nent + p.S - 1) / p.S;
  p.items_max = items_max;
  p.nt_max = split ? (p.items_max + 1) / 2 : p.items_max;
  p.sort_blocks = pairs ? (nent + kSortTile - 1) / kSortTile : 0;
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 1024); return at; };
  const size_t nv = (size_t)nent;
  p.off_Wh = take((size_t)p.nt_max * kTileN * kD * 2);
  p.off_Wl = split ? take((size_t)p.nt_max * kTileN * kD * 2) : 0;
  p.off_pn = take((size_t)p.nt_max * kTileN * 4);
  p.off_caprow = take(nv * 4);
  p.off_vlen = take(nv * 4);
  p.off_ifirst = take((size_t)p.items_max * 4);
  p.off_incap = take((size_t)p.items_max * 4);
  p.off_cpre = take((size_t)(p.items_max + 1) * 4);
  p.off_timg = take((size_t)p.nt_max * 4);
  p.off_iitems = take((size_t)p.nwin * 4);
  p.off_icost = take((size_t)p.nwin * 4);
  p.off_counts = take(256);
  p.off_Ct = take((size_t)Bi * kRRows * kD * 2);
  p.off_Ck = take((size_t)Bi * kD * kRCols * 2);
  p.off_Ctl = split ? take((size_t)Bi * kRRows * kD * 2) : 0;
  p.off_Ckl = split ? take((size_t)Bi * kD * kRCols * 2) : 0;
  p.off_keyA = p.off_valA = p.off_keyB = p.off_valB = p.off_hist = p.off_eoff = p.off_capS = p.off_mS = 0;
  if (pairs) {
    p.off_keyA = take(nv * 4);
    p.off_valA = take(nv * 4);
    p.off_keyB = take(nv * 4);
    p.off_valB = take(nv * 4);
    p.off_hist = take((size_t)p.sort_blocks * 256 * 4);
    p.off_eoff = take((size_t)(Bi + 1) * 4);
    p.off_capS = take(nv * 4);
    p.off_mS = take(nv * 4);
  }
  p.total = o;
  return p;
}

// K candidates per image: at most ceil(K / per_unit) units per image (even in split precision)
static CandPlan make_cand_plan(int Bi, int K, int T, bool split) {
  const int U = split ? 64 : kTileN;
  const long long per_unit = U / ((T + 3) & ~3);   // captions that always fit in one unit
  long long units = (K + per_unit - 1) / per_unit;
  if (split) units += units & 1;                   // whole tiles per image
  return make_plan(Bi, (long long)Bi * K, (long long)Bi * units, T, split, false);
}

// P pairs: image b with n_b > 0 pairs takes at most ceil(n_b / per_unit) units plus one of tile padding in split
// precision, so all of them at most ceil(P / per_unit) + (1 + split) * min(Bi, P)
static CandPlan make_pairs_plan(int Bi, long long P, int T, bool split) {
  const int U = split ? 64 : kTileN;
  const long long per_unit = U / ((T + 3) & ~3);
  const long long items = (P + per_unit - 1) / per_unit + (split ? 2 : 1) * std::min<long long>(Bi, P);
  return make_plan(Bi, P, items, T, split, true);
}

// the cost prefix and the packed row indices are int32
static bool cand_plan_fits(const CandPlan& p) {
  return p.items_max * kMaxItemCost < (long long)INT32_MAX && p.nt_max * kTileN < (long long)INT32_MAX;
}

// cand: the caption index of every entry; eoff: CSR entry offsets of the images, or nullptr for K entries per image.
// m_out[v] is written for every entry v.  v16 / rowst != nullptr (pair training forward): the pair kernels also save
// the normalised context vectors and row statistics of every packed word row for agb_damsm_pairs_bwd.
template <typename T16>
static int run_cand(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                    const int32_t* cap_lens, int Bc, const int32_t* cand, const int32_t* eoff, int Bi, int K, int T,
                    int R, float gamma1, float gamma2, float* m_out, char* ws, const CandPlan& pl, cudaStream_t st,
                    void* v16 = nullptr, float4* rowst = nullptr) {
  const bool bf = std::is_same<T16, __nv_bfloat16>::value;
  const int U = pl.split ? 64 : kTileN;
  T16* Wh = (T16*)(ws + pl.off_Wh);
  T16* Wl = pl.split ? (T16*)(ws + pl.off_Wl) : nullptr;
  float* pn = (float*)(ws + pl.off_pn);
  int32_t* cap_row = (int32_t*)(ws + pl.off_caprow);
  int32_t* vlen = (int32_t*)(ws + pl.off_vlen);
  int32_t* ifirst = (int32_t*)(ws + pl.off_ifirst);
  int32_t* incap = (int32_t*)(ws + pl.off_incap);
  int32_t* cpre = (int32_t*)(ws + pl.off_cpre);
  int32_t* timg = (int32_t*)(ws + pl.off_timg);
  int32_t* iitems = (int32_t*)(ws + pl.off_iitems);
  int32_t* icost = (int32_t*)(ws + pl.off_icost);
  int32_t* ntiles = (int32_t*)(ws + pl.off_counts);
  int32_t* nunits = pl.split ? ntiles + 1 : nullptr;
  T16* Ct = (T16*)(ws + pl.off_Ct);
  T16* Ck = (T16*)(ws + pl.off_Ck);
  T16* Ctl = pl.split ? (T16*)(ws + pl.off_Ctl) : nullptr;
  T16* Ckl = pl.split ? (T16*)(ws + pl.off_Ckl) : nullptr;

  const int nwin = (int)pl.nwin;
  const int pack_blocks = cdiv(nwin, 8);
  cand_pack_kernel<false><<<pack_blocks, 256, 0, st>>>(cap_lens, Bc, T, cand, eoff, Bi, K, nwin, pl.S, U, iitems,
                                                       icost, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
  if (int rc = check_launch("cand_pack_kernel<false>")) return rc;
  cand_scan_kernel<<<1, 1024, 0, st>>>(iitems, icost, nwin, kTileN / U, cpre, ntiles, nunits);
  if (int rc = check_launch("cand_scan_kernel")) return rc;
  cand_pack_kernel<true><<<pack_blocks, 256, 0, st>>>(cap_lens, Bc, T, cand, eoff, Bi, K, nwin, pl.S, U, iitems, icost,
                                                      cap_row, vlen, ifirst, incap, cpre, timg);
  if (int rc = check_launch("cand_pack_kernel<true>")) return rc;
  cand_rows_kernel<T16><<<(unsigned)pl.nt_max, 512, 0, st>>>(words, ws_b, ws_d, ws_t, cand, vlen, cap_row, ifirst, incap,
                                                             U, ntiles, Wh, Wl, pn);
  if (int rc = check_launch("cand_rows_kernel")) return rc;
  pack_img_kernel_tc<T16><<<dim3(kRRows / 32, kD / 32, Bi), dim3(32, 8), 0, st>>>(img, Ck, Ct, Ckl, Ctl, R);
  if (int rc = check_launch("pack_img_kernel_tc")) return rc;

  FwdCandParams p;
  p.tile_first = ifirst; p.tile_ncap = incap; p.ntiles = ntiles; p.cap_row = cap_row; p.cap_lens = vlen;
  p.tile_cpre = cpre;
  p.uniform_split = 0;
  p.img_block = 0;
  p.dup_rem = R > 256 ? 1 : 0;
  p.pn = pn; p.m_out = m_out; p.Bi = Bi; p.Bc = 0; p.T = T; p.R = R;
  p.scale_log2 = kLog2e / sqrtf((float)kD);
  p.g1_log2 = gamma1 * kLog2e;
  p.gamma2 = gamma2;
  p.v16 = v16; p.rowst = rowst; p.Ntot = 0;
  p.tile_img = timg;
  p.wh = Wh;
  const int grid = (int)std::min<long long>(num_sms(), pl.items_max);
  CUtensorMap mapCt, mapCk;
  if (int rc = make_tmap_2d(&mapCt, Ct, (uint64_t)Bi * kRRows, kD, 128, bf)) return rc;
  if (int rc = make_tmap_2d(&mapCk, Ck, (uint64_t)Bi * kD, kRCols, 128, bf)) return rc;
  if (pl.split) {
    if constexpr (std::is_same<T16, __half>::value) {
      CUtensorMap mapWh, mapWl, mapCtl, mapCkl;
      if (int rc = make_tmap_2d(&mapWh, Wh, (uint64_t)pl.nt_max * kTileN, kD, 64, false)) return rc;
      if (int rc = make_tmap_2d(&mapWl, Wl, (uint64_t)pl.nt_max * kTileN, kD, 64, false)) return rc;
      if (int rc = make_tmap_2d(&mapCtl, Ctl, (uint64_t)Bi * kRRows, kD, 128, false)) return rc;
      if (int rc = make_tmap_2d(&mapCkl, Ckl, (uint64_t)Bi * kD, kRCols, 128, false)) return rc;
      FwdXCandParams xp;
      xp.f = p; xp.unit_first = ifirst; xp.unit_ncap = incap; xp.nunits = nunits;
      xp.tile_img = timg; xp.wh = Wh; xp.wl = Wl;
      auto kx = v16 ? damsm_fwd2x_kernel<true, true> : damsm_fwd2x_kernel<false, true>;
      AGB_CUDA(cudaFuncSetAttribute(kx, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes2));
      const int slot = prof_begin(PROF_DAMSM_CAND, st);
      kx<<<grid, kThreads, kSmemBytes2, st>>>(mapWh, mapWl, mapCt, mapCtl, mapCk, mapCkl, xp);
      prof_end(slot, st);
      return check_launch("damsm_fwd2x_kernel<cand>");
    } else {
      return fail_unsupported("split precision needs fp16 operands");
    }
  }
  CUtensorMap mapW;
  if (int rc = make_tmap_2d(&mapW, Wh, (uint64_t)pl.nt_max * kTileN, kD, 128, bf)) return rc;
  auto kern = v16 ? damsm_fwd2_kernel<T16, true, true> : damsm_fwd2_kernel<T16, false, true>;
  AGB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes2));
  const int slot = prof_begin(PROF_DAMSM_CAND, st);
  kern<<<grid, kThreads, kSmemBytes2, st>>>(mapW, mapCt, mapCk, p);
  prof_end(slot, st);
  return check_launch("damsm_fwd2_kernel<cand>");
}

// pair lists: group the pairs by image (two radix passes), CSR offsets, then the candidate pipeline over the
// sorted pairs and a scatter of m back to list order
template <typename T16>
static int run_pairs(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                     const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap, int P,
                     int T, int R, float gamma1, float gamma2, float* m_out, char* ws, const CandPlan& pl,
                     cudaStream_t st, void* v16 = nullptr, float4* rowst = nullptr) {
  int32_t* keyA = (int32_t*)(ws + pl.off_keyA);
  int32_t* valA = (int32_t*)(ws + pl.off_valA);
  int32_t* keyB = (int32_t*)(ws + pl.off_keyB);
  int32_t* valB = (int32_t*)(ws + pl.off_valB);
  int32_t* hist = (int32_t*)(ws + pl.off_hist);
  int32_t* eoff = (int32_t*)(ws + pl.off_eoff);
  int32_t* capS = (int32_t*)(ws + pl.off_capS);
  float* mS = (float*)(ws + pl.off_mS);
  const unsigned G = (unsigned)pl.sort_blocks;
  for (int pass = 0; pass < 2; ++pass) {
    const int32_t* kin = pass ? keyA : nullptr;
    const int32_t* vin = pass ? valA : nullptr;
    int32_t* kout = pass ? keyB : keyA;
    int32_t* vout = pass ? valB : valA;
    pair_hist_kernel<<<G, 256, 0, st>>>(pair_img, Bi, kin, P, 8 * pass, hist);
    if (int rc = check_launch("pair_hist_kernel")) return rc;
    excl_scan_kernel<<<1, 1024, 0, st>>>(hist, (int)(256 * G));
    if (int rc = check_launch("excl_scan_kernel")) return rc;
    pair_scatter_kernel<<<G, 256, 0, st>>>(pair_img, Bi, kin, vin, P, 8 * pass, hist, kout, vout);
    if (int rc = check_launch("pair_scatter_kernel")) return rc;
  }
  pair_offsets_kernel<<<(unsigned)((std::max(P, Bi + 1) + 255LL) / 256), 256, 0, st>>>(keyB, valB, pair_cap, P, Bi, eoff, capS);
  if (int rc = check_launch("pair_offsets_kernel")) return rc;
  if (int rc = run_cand<T16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bc, capS, eoff, Bi, 0, T, R, gamma1, gamma2, mS,
                             ws, pl, st, v16, rowst))
    return rc;
  pair_scatter_m_kernel<<<(unsigned)((P + 255LL) / 256), 256, 0, st>>>(mS, valB, eoff, Bi, P, m_out);
  return check_launch("pair_scatter_m_kernel");
}

#include "damsm_tc_bwd2.inc"
#include "damsm_tc_bwd3.inc"
#include "damsm_tc_bwd2_host.inc"
#include "damsm_tc_pairs_bwd.inc"

}  // namespace tc

int damsm_tc_supported(int T, int D, int R) { return (D == tc::kD && T >= 1 && T <= 32 && R >= 1 && R <= tc::kRCols) ? 1 : 0; }

size_t damsm_tc_workspace_bytes(int Bi, int Bc, int T, int D, int R, int math) {
  return tc::make_tc_plan(Bi, Bc, T, D, R, math == AGB_MATH_TC_F16X2).total;
}

int damsm_tc_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                 const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1, float gamma2,
                 float eps, int row_offset, float* m_out, float* att_out, const float* cnn, const float* rnn,
                 float* scos_out, void* workspace, size_t workspace_bytes, int math, int save, cudaStream_t st) {
  if (Bi <= 0 || Bc <= 0) return fail_arg("non-positive batch");
  if (Bi > 65535) return fail_unsupported("Bi=%d > 65535", Bi);
  if (math != AGB_MATH_TC_BF16 && gamma1 > 11.f) return fail_unsupported("gamma1=%g overflows fp16 (use bf16 or fp32 math)", gamma1);
  const tc::TcPlan pl = tc::make_tc_plan(Bi, Bc, T, D, R, math == AGB_MATH_TC_F16X2);
  if (workspace_bytes < pl.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return AGB_E_WORKSPACE;
  }
  char* ws = (char*)workspace;
  int rc;
  // the matched-pair attention maps and the sentence cosine only read the caller's inputs: they run on a
  // forked stream beside the pack kernels and the pair kernel and join before this call returns
  tc::SideStream* side = nullptr;
  int rc_side = 0;
  if (att_out || cnn) {
    if (att_out && (row_offset < 0 || row_offset + Bi > Bc)) return fail_arg("row_offset=%d out of range", row_offset);
    if ((rc = tc::side_stream(&side))) return rc;
    if ((rc = tc::side_fork(side, st))) return rc;
    if (att_out)
      rc_side = damsm_diag_att_maps(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, T, D, R, gamma1, row_offset, att_out,
                                    (float*)(ws + pl.off_attS), (float*)(ws + pl.off_attB), side->stream);
    if (cnn && rc_side == 0) rc_side = sent_cos_fwd_launch(cnn, rnn, Bi, Bc, D, eps, scos_out, side->stream);
  }
  if (rc_side == 0) {
    if (math == AGB_MATH_TC_BF16)
      rc = tc::run_fwd<__nv_bfloat16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, R, gamma1, gamma2, m_out, ws, pl, save != 0, st);
    else
      rc = tc::run_fwd<__half>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, R, gamma1, gamma2, m_out, ws, pl, save != 0, st);
  } else {
    rc = rc_side;
  }
  // joined on every path after the fork (an enclosing graph capture must not be left forked)
  if (side)
    if (int rj = tc::side_join(side, st)) return rc ? rc : rj;
  return rc;
}

// 0 when the shapes are outside the candidate path's range (the caller has checked T, D, R and math)
size_t damsm_tc_cand_workspace_bytes(int Bi, int K, int T, int math) {
  if (Bi <= 0 || Bi > 65535 || K <= 0 || (long long)Bi * K >= (long long)INT32_MAX) return 0;
  const tc::CandPlan pl = tc::make_cand_plan(Bi, K, T, math == AGB_MATH_TC_F16X2);
  return tc::cand_plan_fits(pl) ? pl.total : 0;
}

int damsm_tc_cand_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                      const int32_t* cap_lens, int Bc, const int32_t* cand, int Bi, int K, int T, int R, float gamma1,
                      float gamma2, float* m_out, void* workspace, size_t workspace_bytes, int math, cudaStream_t st) {
  if (Bc <= 0 || Bi <= 0 || K <= 0) return fail_arg("non-positive size");
  if (Bi > 65535) return fail_unsupported("Bi=%d > 65535", Bi);
  if ((long long)Bi * K >= (long long)INT32_MAX) return fail_unsupported("Bi*K=%lld >= 2^31", (long long)Bi * K);
  if (math != AGB_MATH_TC_BF16 && gamma1 > 11.f) return fail_unsupported("gamma1=%g overflows fp16 (use bf16 math)", gamma1);
  const tc::CandPlan pl = tc::make_cand_plan(Bi, K, T, math == AGB_MATH_TC_F16X2);
  if (!tc::cand_plan_fits(pl)) return fail_unsupported("Bi=%d K=%d: %lld word tiles exceed the int32 cost prefix", Bi, K, pl.nt_max);
  if (workspace_bytes < pl.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return AGB_E_WORKSPACE;
  }
  if (math == AGB_MATH_TC_BF16)
    return tc::run_cand<__nv_bfloat16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bc, cand, nullptr, Bi, K, T, R, gamma1,
                                       gamma2, m_out, (char*)workspace, pl, st);
  return tc::run_cand<__half>(img, words, ws_b, ws_d, ws_t, cap_lens, Bc, cand, nullptr, Bi, K, T, R, gamma1, gamma2,
                              m_out, (char*)workspace, pl, st);
}

// 0 when the shapes are outside the pair path's range (the caller has checked T, D, R and math)
size_t damsm_tc_pairs_workspace_bytes(int Bi, int Bc, long long P, int T, int math) {
  if (Bi <= 0 || Bi > 65535 || Bc <= 0 || P < 0 || P >= (long long)INT32_MAX) return 0;
  const tc::CandPlan pl = tc::make_pairs_plan(Bi, P, T, math == AGB_MATH_TC_F16X2);
  return tc::cand_plan_fits(pl) ? pl.total : 0;
}

int damsm_tc_pairs_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                       const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                       long long P, int T, int D, int R, float gamma1, float gamma2, float* m_out, float* att_out,
                       void* workspace, size_t workspace_bytes, int math, cudaStream_t st) {
  if (Bc <= 0 || Bi <= 0 || P < 0) return fail_arg("non-positive size");
  if (Bi > 65535) return fail_unsupported("Bi=%d > 65535", Bi);
  if (P >= (long long)INT32_MAX) return fail_unsupported("P=%lld >= 2^31", P);
  if (math != AGB_MATH_TC_BF16 && gamma1 > 11.f) return fail_unsupported("gamma1=%g overflows fp16 (use bf16 math)", gamma1);
  const tc::CandPlan pl = tc::make_pairs_plan(Bi, P, T, math == AGB_MATH_TC_F16X2);
  if (!tc::cand_plan_fits(pl)) return fail_unsupported("Bi=%d P=%lld: %lld word tiles exceed the int32 cost prefix", Bi, P, pl.nt_max);
  if (P == 0) return 0;
  if (workspace_bytes < pl.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return AGB_E_WORKSPACE;
  }
  int rc;
  // the pair maps only read the caller's inputs: they run on a forked stream beside the grouping, the pack
  // kernels and the pair kernel, as agb_damsm_fwd runs its matched maps
  tc::SideStream* side = nullptr;
  int rc_side = 0;
  if (att_out) {
    if ((rc = tc::side_stream(&side))) return rc;
    if ((rc = tc::side_fork(side, st))) return rc;
    rc_side = damsm_pair_att_maps(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, (int)P, T, D, R,
                                  gamma1, att_out, side->stream);
  }
  if (rc_side == 0) {
    if (math == AGB_MATH_TC_BF16)
      rc = tc::run_pairs<__nv_bfloat16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, (int)P, T,
                                        R, gamma1, gamma2, m_out, (char*)workspace, pl, st);
    else
      rc = tc::run_pairs<__half>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, (int)P, T, R,
                                 gamma1, gamma2, m_out, (char*)workspace, pl, st);
  } else {
    rc = rc_side;
  }
  // joined on every path after the fork (an enclosing graph capture must not be left forked)
  if (side)
    if (int rj = tc::side_join(side, st)) return rc ? rc : rj;
  return rc;
}

// 0 when the shapes are outside the pair path's range (the caller has checked T, D, R and math)
size_t damsm_tc_pairs_train_workspace_bytes(int Bi, int Bc, long long P, int T, int math) {
  if (Bi <= 0 || Bi > 65535 || Bc <= 0 || P < 0 || P >= (long long)INT32_MAX) return 0;
  const tc::PairTrainPlan pl = tc::make_pairs_train_plan(Bi, Bc, P, T, math == AGB_MATH_TC_F16X2);
  return tc::cand_plan_fits(pl.c) ? pl.total : 0;
}

static int pairs_train_check(int Bi, int Bc, long long P, float gamma1, int math) {
  if (Bc <= 0 || Bi <= 0 || P < 0) return fail_arg("non-positive size");
  if (Bi > 65535) return fail_unsupported("Bi=%d > 65535", Bi);
  if (P >= (long long)INT32_MAX) return fail_unsupported("P=%lld >= 2^31", P);
  if (math != AGB_MATH_TC_BF16 && gamma1 > 11.f) return fail_unsupported("gamma1=%g overflows fp16 (use bf16 math)", gamma1);
  return 0;
}

int damsm_tc_pairs_train_fwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                             const int32_t* cap_lens, int Bi, int Bc, const int32_t* pair_img, const int32_t* pair_cap,
                             long long P, int T, int R, float gamma1, float gamma2, float* m_out, void* workspace,
                             size_t workspace_bytes, int math, cudaStream_t st) {
  if (int rc = pairs_train_check(Bi, Bc, P, gamma1, math)) return rc;
  const tc::PairTrainPlan pl = tc::make_pairs_train_plan(Bi, Bc, P, T, math == AGB_MATH_TC_F16X2);
  if (!tc::cand_plan_fits(pl.c)) return fail_unsupported("Bi=%d P=%lld: %lld word tiles exceed the int32 cost prefix", Bi, P, pl.c.nt_max);
  if (P == 0) return 0;
  if (workspace_bytes < pl.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return AGB_E_WORKSPACE;
  }
  char* ws = (char*)workspace;
  void* v16 = ws + pl.off_v16;
  float4* rowst = (float4*)(ws + pl.off_rowst);
  if (math == AGB_MATH_TC_BF16)
    return tc::run_pairs<__nv_bfloat16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, (int)P, T, R,
                                        gamma1, gamma2, m_out, ws, pl.c, st, v16, rowst);
  return tc::run_pairs<__half>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, pair_img, pair_cap, (int)P, T, R, gamma1,
                               gamma2, m_out, ws, pl.c, st, v16, rowst);
}

int damsm_tc_pairs_bwd(const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t, const int32_t* cap_lens, int Bi,
                       int Bc, long long P, int T, int R, float gamma1, float gamma2, const float* dm, float* dimg,
                       float* dwords, void* workspace, size_t workspace_bytes, int math, cudaStream_t st) {
  if (int rc = pairs_train_check(Bi, Bc, P, gamma1, math)) return rc;
  const tc::PairTrainPlan pl = tc::make_pairs_train_plan(Bi, Bc, P, T, math == AGB_MATH_TC_F16X2);
  if (!tc::cand_plan_fits(pl.c)) return fail_unsupported("Bi=%d P=%lld: %lld word tiles exceed the int32 cost prefix", Bi, P, pl.c.nt_max);
  if (P == 0) {   // no pair: every gradient is zero
    if (dimg) AGB_CUDA(cudaMemsetAsync(dimg, 0, (size_t)Bi * tc::kD * R * sizeof(float), st));
    if (dwords) AGB_CUDA(cudaMemsetAsync(dwords, 0, (size_t)Bc * T * tc::kD * sizeof(float), st));
    return 0;
  }
  if (workspace_bytes < pl.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return AGB_E_WORKSPACE;
  }
  if (math == AGB_MATH_TC_BF16)
    return tc::run_pairs_bwd<__nv_bfloat16>(words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, (int)P, T, R, gamma1, gamma2, dm,
                                            dimg, dwords, (char*)workspace, pl, st);
  return tc::run_pairs_bwd<__half>(words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, (int)P, T, R, gamma1, gamma2, dm, dimg,
                                   dwords, (char*)workspace, pl, st);
}

size_t sent_cos_pairs_bwd_workspace_bytes(int Bi, int Bc, long long P) {
  if (Bi <= 0 || Bc <= 0 || P < 0 || P >= (long long)INT32_MAX) return 0;
  return tc::make_sent_pairs_plan(Bi, Bc, P).total;
}

int sent_cos_pairs_bwd(const float* cnn, const float* rnn, int Bi, int Bc, const int32_t* pair_img,
                       const int32_t* pair_cap, long long P, int D, float eps, const float* dscos, float* dcnn,
                       float* drnn, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (Bi <= 0 || Bc <= 0 || D <= 0 || P < 0) return fail_arg("non-positive size");
  if (P >= (long long)INT32_MAX) return fail_unsupported("P=%lld >= 2^31", P);
  if (P == 0) {
    if (dcnn) AGB_CUDA(cudaMemsetAsync(dcnn, 0, (size_t)Bi * D * sizeof(float), st));
    if (drnn) AGB_CUDA(cudaMemsetAsync(drnn, 0, (size_t)Bc * D * sizeof(float), st));
    return 0;
  }
  const tc::SentPairsPlan pl = tc::make_sent_pairs_plan(Bi, Bc, P);
  if (workspace_bytes < pl.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return AGB_E_WORKSPACE;
  }
  return tc::run_sent_pairs_bwd(cnn, rnn, Bi, Bc, pair_img, pair_cap, (int)P, D, eps, dscos, dcnn, drnn,
                                (char*)workspace, pl, st);
}

int damsm_tc_bwd(const float* img, const float* words, int64_t ws_b, int64_t ws_d, int64_t ws_t,
                 const int32_t* cap_lens, int Bi, int Bc, int T, int D, int R, float gamma1, float gamma2,
                 float eps, const float* dm, const float* m_fwd, const float* gscale, float* dimg, float* dwords,
                 void* workspace, size_t workspace_bytes, int ws_from_fwd, int math, cudaStream_t st) {
  if (Bi <= 0 || Bc <= 0) return fail_arg("non-positive batch");
  if (Bi > 65535) return fail_unsupported("Bi=%d > 65535", Bi);
  const tc::TcPlan pl = tc::make_tc_plan(Bi, Bc, T, D, R, math == AGB_MATH_TC_F16X2);
  if (workspace_bytes < pl.total) {
    set_error("workspace too small: %zu < %zu", workspace_bytes, pl.total);
    return AGB_E_WORKSPACE;
  }
  if (pl.save) {
    if (math == AGB_MATH_TC_BF16)
      return tc::run_bwd3<__nv_bfloat16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, R, gamma1, gamma2, dm, m_fwd,
                                         gscale, dimg, dwords, (char*)workspace, pl, ws_from_fwd, st);
    return tc::run_bwd3<__half>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, R, gamma1, gamma2, dm, m_fwd, gscale,
                                dimg, dwords, (char*)workspace, pl, ws_from_fwd, st);
  }
  if (math == AGB_MATH_TC_BF16)
    return tc::run_bwd2<__nv_bfloat16>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, R, gamma1, gamma2, dm, m_fwd,
                                       gscale, dimg, dwords, (char*)workspace, pl, ws_from_fwd, st);
  return tc::run_bwd2<__half>(img, words, ws_b, ws_d, ws_t, cap_lens, Bi, Bc, T, R, gamma1, gamma2, dm, m_fwd, gscale,
                              dimg, dwords, (char*)workspace, pl, ws_from_fwd, st);
}

}  // namespace agb

#ifdef AGB_TIMELINE
// debug build only (-DAGB_TIMELINE): the clock64 timeline CTA 0 of damsm_bwd3_kernel recorded, and per-CTA run times
extern "C" int agb_damsm_debug_timeline(long long* out, int n) {
  const size_t bytes = std::min((size_t)n * 8, sizeof(agb::tc::g_tl));
  return (int)cudaMemcpyFromSymbol(out, agb::tc::g_tl, bytes);
}
extern "C" int agb_damsm_debug_cta_times(long long* out, int n) {
  const size_t bytes = std::min((size_t)n * 8, sizeof(agb::tc::g_tl_cta));
  return (int)cudaMemcpyFromSymbol(out, agb::tc::g_tl_cta, bytes);
}
#endif
