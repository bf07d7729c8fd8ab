// route.cu -- the exchange step of the item-sharded ingest (SURVEY.md 8e): every GPU holds an arbitrary
// slice of the (row, key, inc) event stream; an event belongs to the GPU that owns its row,
// owner = row mod G, local row = row div G.
//
// One kernel does the partition AND the transfer: k_route_scatter partitions a tile of 4096 events by
// owner in shared memory and writes each owner's run straight into that GPU's receive columns through its
// peer mapping -- NVLink stores in coalesced runs of ~4096 / G events, no intermediate send buffer, no
// sort, no NCCL collective on the data path.  The only collective is the G x G count matrix the callers
// exchange beforehand (a few hundred bytes) so that every source knows where its region starts in every
// destination.
#include "common.cuh"

namespace {

constexpr int R_THREADS = 512;
constexpr int R_ITEMS = 8;
constexpr int R_TILE = R_THREADS * R_ITEMS;

__device__ __forceinline__ void owner_of(long long row, int G, int gmask, int gshift, int& owner, long long& local) {
  if (row < 0) {  // not a row: stays negative at its first destination, where K1 reports it
    owner = 0;
    local = row;
  } else if (gmask >= 0) {
    owner = (int)(row & gmask);
    local = row >> gshift;
  } else {
    local = row / G;
    owner = (int)(row - local * G);
  }
}

__global__ void __launch_bounds__(512) k_route_count(const long long* __restrict__ row, long long n, int G, int gmask,
                                                     int gshift, unsigned long long* __restrict__ counts) {
  __shared__ unsigned hist[16][MB200_MAX_BLOCKS];  // one private histogram per warp
  const int warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 16 * MB200_MAX_BLOCKS; i += blockDim.x) (&hist[0][0])[i] = 0;
  __syncthreads();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
    int o;
    long long l;
    owner_of(__ldg(row + t), G, gmask, gshift, o, l);
    atomicAdd(&hist[warp][o], 1u);
  }
  __syncthreads();
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    unsigned s = 0;
    for (int w = 0; w < 16; w++) s += hist[w][g];
    if (s) atomicAdd(&counts[g], (unsigned long long)s);
  }
}

struct RouteArgs {
  const long long* row;
  const long long* key;
  const float* inc;
  long long n;
  int G, gmask, gshift;
  unsigned long long* cursor;  // [G] next free slot of this source in every destination
  long long* dst_row[MB200_MAX_BLOCKS];
  long long* dst_key[MB200_MAX_BLOCKS];
  float* dst_inc[MB200_MAX_BLOCKS];
};

struct RouteSmem {
  long long st_row[R_TILE];
  long long st_key[R_TILE];
  float st_inc[R_TILE];
  unsigned char st_own[R_TILE];
  unsigned hist[MB200_MAX_BLOCKS];
  unsigned loff[MB200_MAX_BLOCKS];
  unsigned long long gbase[MB200_MAX_BLOCKS];
};

__global__ void __launch_bounds__(R_THREADS, 2) k_route_scatter(const RouteArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  RouteSmem& sm = *reinterpret_cast<RouteSmem*>(smem_raw);
  const int tid = threadIdx.x;
  const long long ntiles = (p.n + R_TILE - 1) / R_TILE;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long base = tile * R_TILE;
    if (tid < p.G) sm.hist[tid] = 0;
    __syncthreads();
    long long lrow[R_ITEMS], key[R_ITEMS];
    float inc[R_ITEMS];
    int own[R_ITEMS];
    unsigned rank[R_ITEMS];
#pragma unroll
    for (int i = 0; i < R_ITEMS; i++) {
      const long long idx = base + (long long)i * R_THREADS + tid;
      own[i] = -1;
      if (idx < p.n) {
        owner_of(__ldg(p.row + idx), p.G, p.gmask, p.gshift, own[i], lrow[i]);
        key[i] = __ldg(p.key + idx);
        inc[i] = __ldg(p.inc + idx);
      }
    }
    // rank inside the tile: lanes of a warp that share an owner take one shared-memory atomic together
#pragma unroll
    for (int i = 0; i < R_ITEMS; i++) {
      const unsigned peers = __match_any_sync(0xffffffffu, own[i]);
      const int leader = __ffs(peers) - 1;
      unsigned b = 0;
      if (own[i] >= 0 && (tid & 31) == leader) b = atomicAdd(&sm.hist[own[i]], (unsigned)__popc(peers));
      b = __shfl_sync(0xffffffffu, b, leader);
      rank[i] = b + __popc(peers & ((1u << (tid & 31)) - 1u));
    }
    __syncthreads();
    if (tid == 0) {
      unsigned run = 0;
      for (int g = 0; g < p.G; g++) {
        sm.loff[g] = run;
        const unsigned c = sm.hist[g];
        if (c) sm.gbase[g] = atomicAdd(&p.cursor[g], (unsigned long long)c) - run;
        run += c;
      }
      sm.hist[0] = run;  // total of the tile
    }
    __syncthreads();
    const unsigned total = sm.hist[0];
#pragma unroll
    for (int i = 0; i < R_ITEMS; i++) {
      if (own[i] >= 0) {
        const unsigned pos = sm.loff[own[i]] + rank[i];
        sm.st_row[pos] = lrow[i];
        sm.st_key[pos] = key[i];
        sm.st_inc[pos] = inc[i];
        sm.st_own[pos] = (unsigned char)own[i];
      }
    }
    __syncthreads();
    for (unsigned pos = tid; pos < total; pos += R_THREADS) {
      const int g = sm.st_own[pos];
      const unsigned long long o = sm.gbase[g] + pos;
      p.dst_row[g][o] = sm.st_row[pos];
      p.dst_key[g][o] = sm.st_key[pos];
      p.dst_inc[g][o] = sm.st_inc[pos];
    }
    __syncthreads();
  }
}

void pow2_of(int G, int& gmask, int& gshift) {
  gmask = -1;
  gshift = 0;
  if ((G & (G - 1)) == 0) {
    gmask = G - 1;
    while ((1 << gshift) < G) gshift++;
  }
}

}  // namespace

extern "C" {

int mb200_route_count(mb200_ctx* ctx, const int64_t* row, int64_t n, int32_t shards, int64_t* counts) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_route_count: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  if (n < 0 || shards <= 0 || shards > MB200_MAX_BLOCKS || !counts || (n > 0 && !row))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_route_count: bad arguments (n=%lld, shards=%d; at most %d shards)",
                      (long long)n, shards, MB200_MAX_BLOCKS);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  void* p;
  MB_CHECK(ws_slot(ctx, WS_ROUTE, 2 * MB200_MAX_BLOCKS * sizeof(unsigned long long), &p));
  unsigned long long* d_counts = (unsigned long long*)p;
  MB_CUDA(ctx, cudaMemsetAsync(d_counts, 0, MB200_MAX_BLOCKS * sizeof(unsigned long long), ctx->stream));
  if (n > 0) {
    int gmask, gshift;
    pow2_of(shards, gmask, gshift);
    ProfScope prof(ctx, MB200_K_ROUTE);
    long long want = ceil_div64(n, 512 * 8);
    const int grid = (int)(want < (long long)ctx->num_sms * 4 ? want : (long long)ctx->num_sms * 4);
    k_route_count<<<grid, 512, 0, ctx->stream>>>((const long long*)row, n, shards, gmask, gshift, d_counts);
    ctx->launches++;
    MB_CUDA(ctx, cudaGetLastError());
  }
  unsigned long long h[MB200_MAX_BLOCKS];
  MB_CUDA(ctx, cudaMemcpyAsync(h, d_counts, shards * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int s = 0; s < shards; s++) counts[s] = (int64_t)h[s];
  return MB200_OK;
}

int mb200_route_scatter(mb200_ctx* ctx, const int64_t* row, const int64_t* key, const float* inc, int64_t n,
                        int32_t shards, void* const* dst_row, void* const* dst_key, void* const* dst_inc,
                        const int64_t* dst_offset) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_route_scatter: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  if (n < 0 || shards <= 0 || shards > MB200_MAX_BLOCKS || !dst_row || !dst_key || !dst_inc || !dst_offset ||
      (n > 0 && (!row || !key || !inc)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_route_scatter: bad arguments");
  if (n == 0) return MB200_OK;
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  void* p;
  MB_CHECK(ws_slot(ctx, WS_ROUTE, 2 * MB200_MAX_BLOCKS * sizeof(unsigned long long), &p));
  unsigned long long* d_cursor = (unsigned long long*)p + MB200_MAX_BLOCKS;
  unsigned long long h[MB200_MAX_BLOCKS];
  RouteArgs a;
  memset(&a, 0, sizeof(a));
  for (int s = 0; s < shards; s++) {
    if (dst_offset[s] < 0) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_route_scatter: negative offset");
    h[s] = (unsigned long long)dst_offset[s];
    a.dst_row[s] = (long long*)dst_row[s];
    a.dst_key[s] = (long long*)dst_key[s];
    a.dst_inc[s] = (float*)dst_inc[s];
  }
  // the cursors ride in pageable host memory: cudaMemcpyAsync stages them before it returns
  MB_CUDA(ctx, cudaMemcpyAsync(d_cursor, h, shards * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
  a.row = (const long long*)row;
  a.key = (const long long*)key;
  a.inc = inc;
  a.n = n;
  a.G = shards;
  pow2_of(shards, a.gmask, a.gshift);
  a.cursor = d_cursor;
  const size_t smem = sizeof(RouteSmem);
  MB_CUDA(ctx, cudaFuncSetAttribute(k_route_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  long long want = ceil_div64(n, R_TILE);
  const int grid = (int)(want < (long long)ctx->num_sms * 2 ? want : (long long)ctx->num_sms * 2);
  {
    ProfScope prof(ctx, MB200_K_ROUTE);
    k_route_scatter<<<grid, R_THREADS, smem, ctx->stream>>>(a);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  return MB200_OK;
}

}  // extern "C"
