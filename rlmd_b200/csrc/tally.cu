// Final-time statistics of the discrete sweeps from a tally of outcome-count
// tuples (include/rlmd_b200.h "tally"; reference: the statistic block of
// {coin,dice,dice_sh}_fixed_final_lev, lev/lev_exp.py:87-104, :545-562, :1168-1185).
//
//   count kernel epilogue  -> hash table (tally.cuh), one insertion per investor
//   finalize               -> the distinct tuples as a dense list (compaction);
//                             across GPUs: every rank publishes its list in
//                             peer-mapped memory, raises a flag, and merges ALL
//                             lists in rank order keeping each tuple at its first
//                             occurrence - the one exchange of a sweep, and every
//                             rank ends with the identical list
//   statistics             -> wealth of every (grid point, tuple) with the count
//                             kernels' own expressions (bit-identical data_T
//                             values), then one cluster per grid point: the four
//                             target ranks from a histogram of log wealth and an
//                             exact sort of one bin (checked; else a weighted 3-level
//                             radix select, 11+11+10 bits of the fp32 key), exact
//                             top / rest split with
//                             tie apportioning, two-pass fp64 moments.  The block
//                             owns its row: no atomics on fp64, so the result does
//                             not depend on scheduling, only on the list order.
//
// Semantics follow rowstats.cu (torch.sort / std_mean / median conventions):
// the tests run both on the same sweeps and compare.
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "tally.cuh"

namespace b200 {

struct BinEntry {
  unsigned long long key, count;
};
static_assert(sizeof(BinEntry) == 16, "one 16-byte vector per bin");

constexpr int MERGE_CHUNK = 2048;     // concat positions per block of the mark / unique kernels
constexpr int EX_FLAG_BYTES = 128;    // uint32 [B200_MAX_PEERS] arrival epochs (+ spare)

struct LogTable {
  double lm[B200_MAX_OUTCOMES][B200_MAX_GRID];
};

// ------------------------------------------------------------- layout
struct TallyLayout {
  long long* header;
  unsigned long long* keysA; uint32_t* countsA; uint64_t capA;
  unsigned long long* ukeys; uint32_t* ucnt;
  float* wbuf; int64_t ldw;
  int64_t list_cap;
  // world > 1
  BinEntry* concat; uint32_t* slot_of;
  unsigned long long* keysB; unsigned long long* countsB; uint32_t* posB; uint64_t capB;
  int32_t* blockcnt; int64_t nblk;
  int64_t bytes;
};

static uint64_t pow2_at_least(uint64_t v) {
  uint64_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

static int plan_ok(const b200_tally_plan* p) {
  B200_REQUIRE(p != nullptr, "tally: plan is NULL");
  B200_REQUIRE(p->rows_cap >= 1 && p->rows_cap < ((int64_t)1 << 32), "tally: rows_cap must be in 1..2^32-1");
  B200_REQUIRE(p->bins_cap >= 1 && p->bins_cap < ((int64_t)1 << 31), "tally: bins_cap must be in 1..2^31-1");
  B200_REQUIRE(p->grid_cap >= 1 && p->grid_cap <= B200_MAX_GRID, "tally: grid_cap must be in 1..%d", B200_MAX_GRID);
  B200_REQUIRE(p->world >= 1 && p->world <= B200_MAX_PEERS, "tally: world must be in 1..%d", B200_MAX_PEERS);
  return 0;
}

static TallyLayout layout(const b200_tally_plan& p, void* base) {
  TallyLayout L;
  memset(&L, 0, sizeof(L));
  char* b = (char*)base;
  int64_t off = 0;
  auto take = [&](int64_t bytes) { char* r = b ? b + off : nullptr; off += (bytes + 255) & ~(int64_t)255; return r; };
  L.header = (long long*)take(TH_WORDS * 8);
  L.capA = pow2_at_least((uint64_t)std::max<int64_t>(2048, 2 * std::min(p.rows_cap, p.bins_cap)));
  L.list_cap = (int64_t)(L.capA / 2);
  L.keysA = (unsigned long long*)take((int64_t)L.capA * 8);
  L.countsA = (uint32_t*)take((int64_t)L.capA * 4);
  L.ukeys = (unsigned long long*)take(p.bins_cap * 8);
  L.ucnt = (uint32_t*)take(p.bins_cap * 4);
  L.ldw = (p.bins_cap + 3) & ~(int64_t)3;
  L.wbuf = (float*)take((int64_t)p.grid_cap * L.ldw * 4);
  if (p.world > 1) {
    const int64_t cat = (int64_t)p.world * L.list_cap;
    L.concat = (BinEntry*)take(cat * 16);
    L.slot_of = (uint32_t*)take(cat * 4);
    L.capB = pow2_at_least((uint64_t)std::max<int64_t>(1024, 2 * std::min(cat, p.bins_cap)));
    L.keysB = (unsigned long long*)take((int64_t)L.capB * 8);
    L.countsB = (unsigned long long*)take((int64_t)L.capB * 8);
    L.posB = (uint32_t*)take((int64_t)L.capB * 4);
    L.nblk = (cat + MERGE_CHUNK - 1) / MERGE_CHUNK;
    L.blockcnt = (int32_t*)take(L.nblk * 4);
  }
  L.bytes = off;
  return L;
}

// exchange buffer of one rank: [flags 128 B][list 0][list 1], a list = 16-byte head (count) + list_cap entries
static int64_t exchange_list_bytes(int64_t list_cap) { return 16 + list_cap * 16; }

int tally_device_view(const b200_tally_plan* plan, void* workspace, int32_t horizon, TallyDev* out) {
  if (int rc = plan_ok(plan)) return rc;
  B200_REQUIRE(workspace != nullptr, "tally: workspace is NULL");
  B200_REQUIRE(horizon <= TALLY_MAX_HORIZON, "tally: horizon must be < 2^%d (use b200_lev_sweep + b200_rowstats)",
               TALLY_COUNT_BITS);
  const TallyLayout L = layout(*plan, workspace);
  out->keys = L.keysA;
  out->counts = L.countsA;
  out->header = L.header;
  out->mask = L.capA - 1;
  return 0;
}

// ---------------------------------------------------------------- reset
__global__ void __launch_bounds__(256)
tally_clear_kernel(unsigned long long* keys, uint32_t* counts32, unsigned long long* counts64, uint32_t* pos,
                   uint64_t cap) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
    keys[i] = TALLY_EMPTY;
    if (counts32) counts32[i] = 0;
    if (counts64) counts64[i] = 0;
    if (pos) pos[i] = 0xffffffffu;
  }
}

// ------------------------------------------------------------ compaction
// Table -> dense list, and the table is left empty for the next sweep.  The append
// order is whatever the scheduler makes it (one atomic per warp); the statistics
// of ONE GPU therefore agree run to run up to the rounding of fp64 sums taken in
// a different order, exactly like b200_rowstats.  The last block to finish
// publishes the count (and, across GPUs, raises this rank's flag at every peer).
struct PeerView {
  BinEntry* list[B200_MAX_PEERS];           // the published list of rank r for this epoch, as mapped here
  long long* list_count[B200_MAX_PEERS];
  uint32_t* flags[B200_MAX_PEERS];
  int32_t world, rank;
  uint32_t epoch;
};

// the (n_1, n_2) box of the keys a thread met, as the running maxima of TH_BOX_ACC
__device__ __forceinline__ void box_add(uint32_t (&b)[4], unsigned long long key) {
  int n1, n2, n3;
  tally_unkey(key, n1, n2, n3);
  b[0] = max(b[0], (uint32_t)(TALLY_MAX_HORIZON - n1)); b[1] = max(b[1], (uint32_t)n1);
  b[2] = max(b[2], (uint32_t)(TALLY_MAX_HORIZON - n2)); b[3] = max(b[3], (uint32_t)n2);
}
// the block's maxima -> one global atomicMax per word into dst[0..3]; every thread of the block calls
__device__ __forceinline__ void box_flush(const uint32_t (&b)[4], long long* dst, uint32_t* s /* shared [4] */) {
  if (threadIdx.x < 4) s[threadIdx.x] = 0;
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint32_t m = __reduce_max_sync(0xffffffffu, b[q]);
    if ((threadIdx.x & 31) == 0 && m != 0u) atomicMax(s + q, m);
  }
  __syncthreads();
  if (threadIdx.x < 4 && s[threadIdx.x] != 0u)
    atomicMax(reinterpret_cast<unsigned long long*>(dst) + threadIdx.x, (unsigned long long)s[threadIdx.x]);
}

constexpr int COMPACT_PER = 8;                    // slots per thread
constexpr int COMPACT_CHUNK = 256 * COMPACT_PER;  // slots per block (the table holds a multiple: capacity >= 2048... see layout)

template <bool MULTI>
__global__ void __launch_bounds__(256)
tally_compact_kernel(TallyDev t, unsigned long long* __restrict__ ukeys, uint32_t* __restrict__ ucnt,
                     int64_t out_cap, const __grid_constant__ PeerView P) {
  __shared__ BinEntry stage[COMPACT_CHUNK];
  __shared__ int n_s;
  __shared__ long long base_s;
  __shared__ uint32_t box_s[4];
  uint32_t box[4] = {0, 0, 0, 0};
  const uint64_t cap = t.mask + 1;
  const uint64_t base = (uint64_t)blockIdx.x * COMPACT_CHUNK;
  if (threadIdx.x == 0) n_s = 0;
  // launched early (one GPU): the table is the count kernel's until it has completed
  pdl_launch_dependents();
  pdl_wait();
  __syncthreads();
  // all of a thread's slots (keys and counts) are requested before the first is looked at:
  // one round trip to memory per block, not one per occupied slot
  unsigned long long key[COMPACT_PER];
  uint32_t cnt[COMPACT_PER];
#pragma unroll
  for (int u = 0; u < COMPACT_PER; ++u) {
    const uint64_t i = base + (uint64_t)u * 256 + threadIdx.x;
    key[u] = i < cap ? __ldcg(t.keys + i) : TALLY_EMPTY;
    cnt[u] = i < cap ? __ldcg(t.counts + i) : 0u;
  }
#pragma unroll
  for (int u = 0; u < COMPACT_PER; ++u) {
    if (key[u] == TALLY_EMPTY) continue;
    const uint64_t i = base + (uint64_t)u * 256 + threadIdx.x;
    t.keys[i] = TALLY_EMPTY;
    t.counts[i] = 0;
    if (!MULTI) box_add(box, key[u]);   // (across GPUs the merged list's box is taken by the unique kernel)
    const int p = atomicAdd(&n_s, 1);
    stage[p].key = key[u];
    stage[p].count = cnt[u];
  }
  __syncthreads();
  const int n = n_s;
  if (!MULTI && n > 0) box_flush(box, t.header + TH_BOX_ACC, box_s);
  if (n > 0) {   // one reservation per block
    if (threadIdx.x == 0)
      base_s = (long long)atomicAdd(reinterpret_cast<unsigned long long*>(t.header + TH_LISTPOS), (unsigned long long)n);
    __syncthreads();
    BinEntry* list = MULTI ? P.list[P.rank] : nullptr;
    for (int j = threadIdx.x; j < n; j += 256) {
      const long long p = base_s + j;
      if (p < out_cap) {
        if (MULTI) list[p] = stage[j];
        else { ukeys[p] = stage[j].key; ucnt[p] = (uint32_t)stage[j].count; }
      } else {
        t.header[TH_OVERFLOW] = 1;
      }
    }
  }
  // last block done?
  __shared__ int last_s;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long tk = atomicAdd(reinterpret_cast<unsigned long long*>(t.header + TH_TICKET), 1ull);
    last_s = tk == (unsigned long long)gridDim.x - 1;
  }
  __syncthreads();
  if (!last_s) return;
  __threadfence();
  if (threadIdx.x == 0) {
    const long long total = *reinterpret_cast<volatile long long*>(t.header + TH_LISTPOS);
    const long long m = total < out_cap ? total : out_cap;
    t.header[TH_LISTPOS] = 0;
    t.header[TH_TICKET] = 0;
    if (MULTI) *P.list_count[P.rank] = m;
    else {
      t.header[TH_NBINS] = m;
      t.header[TH_RADIX] = 0;
      for (int q = 0; q < 4; ++q) {
        t.header[TH_BOX + q] = *reinterpret_cast<volatile long long*>(t.header + TH_BOX_ACC + q);
        t.header[TH_BOX_ACC + q] = 0;
      }
    }
  }
  if (MULTI) {
    __syncthreads();
    if (threadIdx.x < P.world && threadIdx.x != P.rank) {
      __threadfence_system();
      uint32_t* f = P.flags[threadIdx.x] + P.rank;
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(P.epoch) : "memory");
    }
  }
}

// ------------------------------------------------------------------ merge
__device__ __forceinline__ void ld_sys_entry(const BinEntry* p, unsigned long long& k, unsigned long long& c) {
  asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(k), "=l"(c) : "l"(p));
}

// Every block waits for the world's flags (one lane per peer), then the grid walks
// the concatenation of the ranks' lists: entry p is copied to local memory and
// added to table B, which also keeps the smallest p of every tuple.
__global__ void __launch_bounds__(256)
tally_merge_kernel(const __grid_constant__ PeerView P, long long* __restrict__ header, BinEntry* __restrict__ concat,
                   uint32_t* __restrict__ slot_of, unsigned long long* __restrict__ keysB,
                   unsigned long long* __restrict__ countsB, uint32_t* __restrict__ posB, uint64_t capB,
                   int64_t concat_cap) {
  __shared__ long long off_s[B200_MAX_PEERS + 1];
  __shared__ int ok_s;
  if (threadIdx.x == 0) ok_s = 1;
  __syncthreads();
  if (threadIdx.x < P.world && threadIdx.x != P.rank) {
    const uint32_t* f = P.flags[P.rank] + threadIdx.x;
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if ((int32_t)(v - P.epoch) >= 0) break;
      __nanosleep(100);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 30000000000ull) { ok_s = 0; break; }
    }
  }
  __syncthreads();
  if (!ok_s) {
    if (threadIdx.x == 0) { header[TH_TIMEOUT] = 1; header[TH_CONCAT] = 0; }
    return;
  }
  if (threadIdx.x == 0) {
    long long acc = 0;
    for (int r = 0; r < P.world; ++r) {
      off_s[r] = acc;
      long long c;
      asm volatile("ld.relaxed.sys.global.s64 %0, [%1];" : "=l"(c) : "l"(P.list_count[r]));
      acc += c;
    }
    off_s[P.world] = acc;
  }
  __syncthreads();
  long long total = off_s[P.world];
  if (total > concat_cap) total = concat_cap;   // cannot happen: every list is <= list_cap
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    header[TH_CONCAT] = total;
    header[TH_RADIX] = 0;
    for (int q = 0; q < 4; ++q) header[TH_BOX + q] = 0;   // filled by tally_unique_kernel (stream order)
  }
  // the part of table B this merge uses: a power of two >= 2 * total (every slot of B is empty between merges)
  uint64_t used = 1024;
  while (used < 2 * (uint64_t)total && used < capB) used <<= 1;
  const uint64_t mask = used - 1;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total;
       p += (long long)gridDim.x * blockDim.x) {
    int r = 0;
    while (r + 1 < P.world && p >= off_s[r + 1]) ++r;
    unsigned long long key, cnt;
    ld_sys_entry(P.list[r] + (p - off_s[r]), key, cnt);
    concat[p].key = key;
    concat[p].count = cnt;
    // insert into B (sized for a load of at most 1/2: a long walk means it is overfull)
    uint32_t found = 0xffffffffu;
    {
      uint64_t slot = tally_mix(key) & mask;
      for (int probe = 0; probe < TALLY_MAX_PROBE; ++probe) {
        unsigned long long cur = __ldcg(keysB + slot);
        if (cur == TALLY_EMPTY) {
          cur = atomicCAS(keysB + slot, TALLY_EMPTY, key);
          if (cur == TALLY_EMPTY) cur = key;
        }
        if (cur == key) {
          atomicAdd(countsB + slot, cnt);
          atomicMin(posB + slot, (uint32_t)p);
          found = (uint32_t)slot;
          break;
        }
        slot = (slot + 1) & mask;
      }
      if (found == 0xffffffffu) header[TH_OVERFLOW] = 1;
    }
    slot_of[p] = found;
  }
}

// first occurrences per chunk of MERGE_CHUNK positions (the grid strides over the chunks: the number of
// bins is only known on the device, and thousands of blocks that find nothing to do cost microseconds)
__global__ void __launch_bounds__(256)
tally_mark_kernel(const long long* __restrict__ header, const uint32_t* __restrict__ slot_of,
                  const uint32_t* __restrict__ posB, int32_t* __restrict__ blockcnt) {
  __shared__ long long red[32];
  const long long total = header[TH_CONCAT];
  const long long nchunks = (total + MERGE_CHUNK - 1) / MERGE_CHUNK;
  for (long long j = blockIdx.x; j < nchunks; j += gridDim.x) {
    const long long base = j * MERGE_CHUNK;
    long long c = 0;
    for (int u = 0; u < MERGE_CHUNK / 256; ++u) {
      const long long p = base + (long long)threadIdx.x * (MERGE_CHUNK / 256) + u;
      if (p < total) {
        const uint32_t s = slot_of[p];
        c += (s != 0xffffffffu && __ldcg(posB + s) == (uint32_t)p);
      }
    }
    c = block_sum(c, red);
    if (threadIdx.x == 0) blockcnt[j] = (int32_t)c;
    __syncthreads();
  }
}

// Stable compaction of the first occurrences: the merged list in concatenation order
// (identical on every rank); table B is emptied on the way.
__global__ void __launch_bounds__(256)
tally_unique_kernel(long long* __restrict__ header, const BinEntry* __restrict__ concat,
                    const uint32_t* __restrict__ slot_of, unsigned long long* __restrict__ keysB,
                    unsigned long long* __restrict__ countsB, uint32_t* __restrict__ posB,
                    const int32_t* __restrict__ blockcnt, unsigned long long* __restrict__ ukeys,
                    uint32_t* __restrict__ ucnt, int64_t bins_cap) {
  __shared__ long long red[32];
  __shared__ long long warp_tot[8];
  __shared__ long long base_s;
  __shared__ uint32_t box_s[4];
  uint32_t box[4] = {0, 0, 0, 0};
  const long long total = header[TH_CONCAT];
  const long long nchunks = (total + MERGE_CHUNK - 1) / MERGE_CHUNK;
  if (total == 0 && blockIdx.x == 0 && threadIdx.x == 0) header[TH_NBINS] = 0;
  for (long long j = blockIdx.x; j < nchunks; j += gridDim.x) {
    const long long base = j * MERGE_CHUNK;
    long long before = 0;
    for (long long i = threadIdx.x; i < j; i += 256) before += blockcnt[i];
    before = block_sum(before, red);
    if (threadIdx.x == 0) base_s = before;
    constexpr int PER = MERGE_CHUNK / 256;
    bool rep[PER];
    uint32_t slot[PER];
    int mine = 0;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const long long p = base + (long long)threadIdx.x * PER + u;
      rep[u] = false;
      slot[u] = 0xffffffffu;
      if (p < total) {
        slot[u] = slot_of[p];
        rep[u] = slot[u] != 0xffffffffu && __ldcg(posB + slot[u]) == (uint32_t)p;
      }
      mine += rep[u];
    }
    // exclusive scan of `mine` over the block
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long up = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += up;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    long long pre = 0, blocktotal = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      if (w < wid) pre += warp_tot[w];
      blocktotal += warp_tot[w];
    }
    long long outp = base_s + pre + incl - mine;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      if (!rep[u]) continue;
      const long long p = base + (long long)threadIdx.x * PER + u;
      if (outp < bins_cap) {
        box_add(box, concat[p].key);
        ukeys[outp] = concat[p].key;
        ucnt[outp] = (uint32_t)__ldcg(countsB + slot[u]);
      } else {
        header[TH_OVERFLOW] = 1;
      }
      keysB[slot[u]] = TALLY_EMPTY;
      countsB[slot[u]] = 0;
      posB[slot[u]] = 0xffffffffu;
      ++outp;
    }
    if (base + MERGE_CHUNK >= total && threadIdx.x == 0) {
      const long long n = base_s + blocktotal;
      header[TH_NBINS] = n < bins_cap ? n : bins_cap;
    }
    __syncthreads();
  }
  box_flush(box, header + TH_BOX, box_s);
}

// ----------------------------------------------------------------- select
// One thread-block CLUSTER per grid point: the bins are split over the cluster's
// CTAs (each keeps its slice's wealth and counts in shared memory after the first
// pass), the radix histograms live in the leader CTA's shared memory and are fed by
// all CTAs through distributed-shared-memory atomics, the fp64 partial sums of the
// CTAs are handed to the leader and added in rank order.  Three cluster barriers per
// pass; no global-memory traffic after the first pass, no atomics on fp64.
constexpr int SEL_THREADS = 1024;
constexpr int SL1 = 2048, SL2 = 2048, SL3 = 1024;   // bins per level (11 + 11 + 10 key bits)
constexpr int SEL_MAX_CLUSTER = 16;                 // > 8: non-portable cluster sizes (B200 allows 16)

// In-place inclusive scans: group `grp` (256 threads) scans histogram `grp` of
// `bins` counters (bins % 256 == 0); groups >= n_hist idle.  Two barriers.
__device__ __forceinline__ void scan_hists(uint32_t* hist, int bins, int n_hist, uint32_t* warp_tot /*[32]*/) {
  const int grp = threadIdx.x >> 8, t = threadIdx.x & 255;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int per = bins >> 8;
  uint32_t* h = hist + grp * bins + t * per;
  uint32_t local = 0;
  if (grp < n_hist)
    for (int i = 0; i < per; ++i) local += h[i];
  uint32_t incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += up;
  }
  if (lane == 31) warp_tot[wid] = incl;
  __syncthreads();
  uint32_t pre = 0;
  for (int w = grp * 8; w < wid; ++w) pre += warp_tot[w];
  uint32_t run = pre + incl - local;
  if (grp < n_hist)
    for (int i = 0; i < per; ++i) { run += h[i]; h[i] = run; }
  __syncthreads();
}

// smallest bin whose inclusive prefix exceeds `rank`; rem = rank inside that bin
__device__ __forceinline__ void find_rank(const uint32_t* pre, int bins, long long rank, int& bin, long long& rem) {
  int lo = 0, hi = bins - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((long long)pre[mid] > rank) hi = mid; else lo = mid + 1;
  }
  bin = lo;
  rem = rank - (lo > 0 ? (long long)pre[lo - 1] : 0);
}

// (grouped shared-memory histogram adds: warp_hist_add, common.cuh)
// The pass's histograms were filled in every CTA's OWN shared memory; the other CTAs now
// add their non-empty bins to the leader's copy (few remote atomics instead of one per element).
__device__ __forceinline__ void push_hist(uint32_t* mine, uint32_t* leaders, int bins, int rank) {
  __syncthreads();
  if (rank != 0)
    for (int i = threadIdx.x; i < bins; i += blockDim.x) {
      const uint32_t v = mine[i];
      if (v != 0u) atomicAdd(leaders + i, v);
    }
}

// Log-wealth route: the candidates of a target (the bins of its log-wealth bin) in the leader's `hist`
constexpr int CAND = 512;                           // per target; more sends the grid point to the radix route
constexpr int CAND_CTA = 256;                       // per target and CTA; more counts as more than CAND

struct SelShared {
  uint32_t hist[4 * SL2];                 // leader: level 1 [0,2048); level 2: 4 x 2048; level 3: 4 x 1024;
                                          // log-wealth route: bin histogram, then candidates [key 4 x CAND |
                                          // count 4 x CAND | the same sorted by (key, count)]
  uint32_t ext[4][2];                     // leader, log-wealth route: max key below / min key above a target's bin
  uint32_t ext_cta[4][2];                 // the same over this CTA's slice
  uint32_t cand_cta[2][4][CAND_CTA];          // log-wealth route: this CTA's candidates (key, count) per target
  int ncand_cta[4], base_cta[4];
  uint32_t sel[4];                        // leader, log-wealth route: the targets' keys
  int ncand[4], found[4], lat_ok;
  double part_d[SEL_MAX_CLUSTER][6];      // leader: the CTAs' partial sums of the running pass
  long long part_i[SEL_MAX_CLUSTER][5];
  double res_d[4];                        // leader: mean_all, mean_top, mean_adj
  long long res_i[16];                    // leader: nonfinite[3], has_nan[3], ties_top, ties_adj, bins[4], rems[4]
  uint32_t warp_tot[32];
  double red_d[32];
  double red_d2[32 * 7];
  long long red_i[32];
};

// sum of N doubles over the block in one go (thread 0 holds the result): one barrier pair for all of them
template <int N>
__device__ __forceinline__ void block_sum_n(double (&v)[N], double* scratch /* >= 32 * N */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < N; ++q) v[q] = warp_sum(v[q]);
  __syncthreads();
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < N; ++q) scratch[q * 32 + wid] = v[q];
  __syncthreads();
  if (wid == 0) {
#pragma unroll
    for (int q = 0; q < N; ++q) {
      const double x = lane < (int)(blockDim.x >> 5) ? scratch[q * 32 + lane] : 0.0;
      v[q] = warp_sum(x);
    }
  }
}

template <int NK>
__global__ void __launch_bounds__(SEL_THREADS)
tally_select_kernel(long long* __restrict__ header, const unsigned long long* __restrict__ ukeys,
                    const uint32_t* __restrict__ ucnt, float* __restrict__ wbuf, int64_t ldw, int32_t H,
                    const __grid_constant__ LogTable lf, double logV0, int64_t n_total, int64_t top,
                    double* __restrict__ stats, int32_t SEL_CACHE /* bins per CTA kept in shared memory */,
                    int32_t force_radix) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int C = (int)cluster.num_blocks(), r = (int)cluster.block_rank();
  __shared__ SelShared sh;
  extern __shared__ __align__(16) uint8_t dyn[];
  float* cw = reinterpret_cast<float*>(dyn);                   // [SEL_CACHE] wealth of the slice's bins beyond the registers
  uint32_t* cc = reinterpret_cast<uint32_t*>(dyn) + SEL_CACHE; // [SEL_CACHE] their counts
  uint16_t* cb = reinterpret_cast<uint16_t*>(cc + SEL_CACHE);  // [SEL_CACHE] their log-wealth bins
  SelShared* L = cluster.map_shared_rank(&sh, 0);              // the leader's copy
  // Launched early (one GPU, depth 1), the select waits here for the compaction's list and header; the next
  // sweep's count kernel may then start on the SMs this grid leaves free (it waits for this grid before it
  // touches the table).
  pdl_launch_dependents();
  pdl_wait();

  const int g = blockIdx.x / C;
  const long long B = header[TH_NBINS];
  const long long n = n_total, K = top;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  double* s = stats + (int64_t)g * 12;
  if (header[TH_TIMEOUT] != 0 || header[TH_OVERFLOW] != 0) {   // uniform over the cluster: nobody touches remote memory
    if (r == 0 && threadIdx.x < 12) s[threadIdx.x] = qnan;
    return;
  }
  const int tid = threadIdx.x, lane = threadIdx.x & 31;
#ifdef B200_TALLY_DEBUG
  int stamp_i = 0;
#define STAMP() do { if (r == 0 && tid == 0 && (g == 0 || g == (int)(gridDim.x / C) - 1)) { header[TH_DEBUG + (g == 0 ? 0 : 24) + stamp_i++] = clock64(); } } while (0)
#else
#define STAMP() do {} while (0)
#endif
  STAMP();
  // this CTA's slice of the bins
  const long long per = (((B + C - 1) / C) + 3) & ~3LL;
  const long long lo = min(B, (long long)r * per), hi = min(B, lo + per);
  const int m = (int)(hi - lo);
  float* __restrict__ w = wbuf + (int64_t)g * ldw + lo;      // spill space for bins beyond the shared-memory cache
  const uint32_t* __restrict__ cnt = ucnt + lo;
  constexpr int REGS = 0;
  double lm[NK];
#pragma unroll
  for (int k = 0; k < NK; ++k) lm[k] = lf.lm[k][g];
  // The log wealth of a bin: the epilogue of the LOG count kernels (lev_sweep.cu) expression for expression,
  // so fl32(exp(lw)) is bit-identical to the data_T entry of every investor in the bin.
  auto lw_of = [&](unsigned long long key) {
    int n1, n2, n3;
    tally_unkey(key, n1, n2, n3);
    int nk[4];
    nk[1] = n1; nk[2] = NK >= 3 ? n2 : 0; nk[3] = NK >= 4 ? n3 : 0;
    nk[0] = H - nk[1] - nk[2] - nk[3];
    double lw = logV0;
#pragma unroll
    for (int k = 0; k < NK; ++k)
      if (nk[k] > 0) lw += (double)nk[k] * lm[k];
    return lw;
  };
  // Log-wealth route (K <= 3, finite log factors): log wealth is linear in the count tuple, so over the
  // (n_1, n_2) box of the list it lies between the values at the box's corners.  SL1 equal bins of log wealth
  // over that range take the place of the radix levels: fl32(exp(.)) is monotone, so the bins are ordered by
  // wealth and a target lies in ONE bin of a few dozen tuples, which the leader then sorts exactly.  Every
  // step is checked on the fp32 values; a grid point that fails a check takes the radix route.
  bool lat = false;
  double lw_lo = 0.0, lw_scale = 0.0;
  if (NK <= 3 && !force_radix) {
    const long long M = TALLY_MAX_HORIZON;
    const long long a[2] = {M - header[TH_BOX + 0], header[TH_BOX + 1]}, b[2] = {M - header[TH_BOX + 2], header[TH_BOX + 3]};
    bool fin = a[0] <= a[1] && b[0] <= b[1];
#pragma unroll
    for (int k = 0; k < NK; ++k) fin = fin && isfinite(lm[k]);
    if (fin) {
      double lo_ = INFINITY, hi_ = -INFINITY;
      for (int u = 0; u < 4; ++u) {
        const double n1 = (double)a[u & 1], n2 = NK >= 3 ? (double)b[u >> 1] : 0.0;
        double v = logV0 + ((double)H - n1 - n2) * lm[0] + n1 * lm[1];
        if (NK >= 3) v += n2 * lm[NK >= 3 ? 2 : 0];
        lo_ = fmin(lo_, v);
        hi_ = fmax(hi_, v);
      }
      if (hi_ > lo_ && isfinite(hi_ - lo_)) { lat = true; lw_lo = lo_; lw_scale = (double)SL1 / (hi_ - lo_); }
    }
  }
  auto lw_bin = [&](double lw) -> uint32_t {   // monotone in lw; out-of-range rounding is clamped
    const double t = (lw - lw_lo) * lw_scale;
    return t >= (double)(SL1 - 1) ? (uint32_t)(SL1 - 1) : t > 0.0 ? (uint32_t)t : 0u;
  };
  if (lat) {
    for (int i = tid; i < SL1; i += SEL_THREADS) sh.hist[i] = 0;
    cluster.sync();
  }
  // The wealth of this grid point at every bin of the slice, formed once and kept in shared memory for the
  // passes; on the log-wealth route the loop also takes pass 0's sums and the bin histogram.
  double a0 = 0;
  long long c0 = 0, pinf = 0;
  for (int i = tid; i < m; i += SEL_THREADS) {
    const double lw = lw_of(__ldg(ukeys + lo + i));
    const float x = (float)exp(lw);
    const uint32_t c = __ldg(cnt + i);
    if (i < SEL_CACHE) { cw[i] = x; cc[i] = c; }
    else w[i] = x;
    if (lat) {
      const uint32_t bn = lw_bin(lw);
      if (i < SEL_CACHE) cb[i] = (uint16_t)bn;
      atomicAdd(sh.hist + bn, c);
      a0 += (double)c * (double)x;
      c0 += c;
      if (isinf(x)) pinf += c;
    }
  }
  __syncthreads();
  auto far_w = [&](int i) { return i < REGS + SEL_CACHE ? cw[i - REGS] : w[i]; };
  auto far_c = [&](int i) { return i < REGS + SEL_CACHE ? cc[i - REGS] : cnt[i]; };
  auto far_b = [&](int i) { return i < SEL_CACHE ? (uint32_t)cb[i] : lw_bin(lw_of(__ldg(ukeys + lo + i))); };
  // f(x, c, in): called by every lane of a warp together (`in` = this lane holds an element)
  auto sweep = [&](auto&& f) {
    for (int base = (tid & ~31); base < m; base += SEL_THREADS) {
      const int i = base + lane;
      const bool in = i < m;
      f(in ? far_w(i) : 0.f, in ? far_c(i) : 0u, in);
    }
  };
  const long long ranks[4] = {(n - 1) / 2, n - K, n - K + (K - 1) / 2, (n - K - 1) / 2};
  uint32_t key_j[4];
  bool radix = !lat;

  if (lat) {
    STAMP();
    // ---- pass 0: sums and the log-wealth histogram are in; the leader finds the targets' bins
    push_hist(sh.hist, L->hist, SL1, r);
    {
      double v[3] = {a0, (double)c0, (double)pinf};   // (counts < 2^32: exact in fp64)
      block_sum_n<3>(v, sh.red_d2);
      if (tid == 0) { L->part_d[r][0] = v[0]; L->part_i[r][0] = (long long)v[1]; L->part_i[r][1] = (long long)v[2]; }
    }
    if (tid < 4) { sh.ext_cta[tid][0] = 0u; sh.ext_cta[tid][1] = 0xffffffffu; sh.ncand_cta[tid] = 0; }
    cluster.sync();
    STAMP();
    if (r == 0) {
      if (tid == 0) {
        double sum_all = 0;
        long long cnt_all = 0, inf_all = 0;
        for (int q = 0; q < C; ++q) { sum_all += sh.part_d[q][0]; cnt_all += sh.part_i[q][0]; inf_all += sh.part_i[q][1]; }
        if (cnt_all != n) header[TH_MISMATCH] = 1;
        // finite log factors: no NaN and no -inf wealth, +inf where exp overflows fp32
        sh.res_i[0] = inf_all > 0; sh.res_i[1] = inf_all > 0; sh.res_i[2] = inf_all > K;
        sh.res_i[3] = 0; sh.res_i[4] = 0; sh.res_i[5] = 0;
        sh.res_d[0] = sum_all / (double)n;
      }
      if (tid < 4) { sh.ncand[tid] = 0; sh.found[tid] = 0; sh.ext[tid][0] = 0u; sh.ext[tid][1] = 0xffffffffu; }
      scan_hists(sh.hist, SL1, 1, sh.warp_tot);
      if (tid < 4) {
        int bin; long long rem;
        find_rank(sh.hist, SL1, ranks[tid], bin, rem);
        sh.res_i[8 + tid] = bin; sh.res_i[12 + tid] = rem;
      }
    }
    cluster.sync();
    STAMP();
    // ---- gather: the tuples of the targets' bins go to the leader (once per distinct bin: targets that share
    // a bin share its list); the sums on either side of thr's bin and the extreme keys on either side of every
    // target's bin are taken on the way
    int bq[4], rep[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      bq[j] = (int)L->res_i[8 + j];
      rep[j] = j;
#pragma unroll
      for (int q = 3; q >= 0; --q)
        if (q < j && bq[q] == bq[j]) rep[j] = q;
    }
    {
      // beside thr's bin the saturated values (+inf, 0) are counted apart: they are thr's ties if thr is one
      double v[7] = {0, 0, 0, 0, 0, 0, 0};   // sum > , sum < thr's bin; count >; +inf >, 0 >, +inf <, 0 <
      uint32_t ext_lo[4] = {0u, 0u, 0u, 0u}, ext_hi[4] = {~0u, ~0u, ~0u, ~0u};
      for (int i = tid; i < m; i += SEL_THREADS) {
        const int bn = (int)far_b(i);
        const float x = far_w(i);
        const uint32_t c = far_c(i), k = float_key(x);
        if (bn > bq[1]) {
          if (isinf(x)) v[3] += (double)c;
          else if (x == 0.f) v[4] += (double)c;
          else { v[0] += (double)c * (double)x; v[2] += (double)c; }
        } else if (bn < bq[1]) {
          if (isinf(x)) v[5] += (double)c;
          else if (x == 0.f) v[6] += (double)c;
          else v[1] += (double)c * (double)x;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (bn < bq[j]) ext_lo[j] = max(ext_lo[j], k);
          else if (bn > bq[j]) ext_hi[j] = min(ext_hi[j], k);
          else if (rep[j] == j) {
            const int p = atomicAdd(&sh.ncand_cta[j], 1);
            if (p < CAND_CTA) { sh.cand_cta[0][j][p] = k; sh.cand_cta[1][j][p] = c; }
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t a = __reduce_max_sync(0xffffffffu, ext_lo[j]), b = __reduce_min_sync(0xffffffffu, ext_hi[j]);
        if (lane == 0) { atomicMax(&sh.ext_cta[j][0], a); atomicMin(&sh.ext_cta[j][1], b); }
      }
      STAMP();
      block_sum_n<7>(v, sh.red_d2);      // (its barriers also close this CTA's extremes)
      if (tid == 0) {
        L->part_d[r][0] = v[0]; L->part_d[r][1] = v[1];
#pragma unroll
        for (int q = 0; q < 5; ++q) L->part_i[r][q] = (long long)v[2 + q];
      }
      if (tid < 8) {
        const int j = tid >> 1;
        if (tid & 1) atomicMin(&L->ext[j][1], sh.ext_cta[j][1]);
        else atomicMax(&L->ext[j][0], sh.ext_cta[j][0]);
      }
      // one reservation per CTA and list in the leader's lists, then plain remote stores
      if (tid < 4 && rep[tid] == tid)
        sh.base_cta[tid] = atomicAdd(&L->ncand[tid], sh.ncand_cta[tid] <= CAND_CTA ? sh.ncand_cta[tid] : CAND + 1);
      __syncthreads();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (rep[j] != j) continue;
        const int nl = min(sh.ncand_cta[j], CAND_CTA), b0 = sh.base_cta[j];
        for (int p = tid; p < nl && b0 + p < CAND; p += SEL_THREADS) {
          L->hist[j * CAND + b0 + p] = sh.cand_cta[0][j][p];
          L->hist[4 * CAND + j * CAND + b0 + p] = sh.cand_cta[1][j][p];
        }
      }
    }
    cluster.sync();
    STAMP();
    if (r == 0) {
      // The candidates of every distinct bin in (key, count) order, eight lanes per candidate: a target is the
      // key whose run of weights covers the rank left inside its bin, and the sums over the sorted copy do not
      // depend on the order in which the CTAs appended them.
      int mq[4], off[5];
      off[0] = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) { mq[j] = rep[j] == j ? min(sh.ncand[j], CAND) : 0; off[j + 1] = off[j] + mq[j]; }
      const int gi = tid >> 3, sub = tid & 7;
      for (int c0 = 0; c0 < off[4]; c0 += SEL_THREADS / 8) {     // the same trip count for every thread
        const int idx = c0 + gi;
        const bool in = idx < off[4];
        int j = 0, oj = 0, mj = mq[0], pos = 0;   // the list of candidate idx (the last with off <= idx: not empty)
#pragma unroll
        for (int q = 1; q < 4; ++q)
          if (idx >= off[q]) { j = q; oj = off[q]; mj = mq[q]; }
        const int t = idx - oj;
        uint32_t kt = 0, ct = 0;
        long long below = 0, eq = 0;
        if (in) {
          const uint32_t* ck = sh.hist + j * CAND;
          const uint32_t* ccn = sh.hist + 4 * CAND + j * CAND;
          kt = ck[t]; ct = ccn[t];
          for (int u = sub; u < mj; u += 8) {
            const uint32_t ku = ck[u], cu = ccn[u];
            if (ku < kt) below += cu;
            else if (ku == kt) eq += cu;
            pos += ku < kt || (ku == kt && (cu < ct || (cu == ct && u < t)));
          }
        }
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
          below += __shfl_xor_sync(0xffffffffu, below, o);
          eq += __shfl_xor_sync(0xffffffffu, eq, o);
          pos += __shfl_xor_sync(0xffffffffu, pos, o);
        }
        if (in && sub == 0) {
          sh.hist[8 * CAND + j * CAND + pos] = kt;
          sh.hist[12 * CAND + j * CAND + pos] = ct;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const long long rem = sh.res_i[12 + q];
            if (rep[q] == j && below <= rem && rem < below + eq) { sh.sel[q] = kt; sh.found[q] = 1; }   // (ties write the same)
          }
        }
      }
      __syncthreads();
      // thr's bin: the exact split of its tuples, as in the radix route's last level
      const uint32_t thr_key = sh.sel[1];
      const int m1 = rep[1] == 0 ? mq[0] : mq[1];
      double f[5] = {0, 0, 0, 0, 0};      // sum > thr, sum < thr, count > thr, count < thr, count of the bin
      for (int t = tid; t < m1; t += SEL_THREADS) {
        const uint32_t k = sh.hist[8 * CAND + rep[1] * CAND + t];
        const long long c = sh.hist[12 * CAND + rep[1] * CAND + t];
        f[4] += (double)c;
        if (k == thr_key) continue;
        const double val = (double)c * (double)key_float(k);
        if (k > thr_key) { f[0] += val; f[2] += (double)c; } else { f[1] += val; f[3] += (double)c; }
      }
      block_sum_n<5>(f, sh.red_d2);
      if (tid == 0) {
        // The bins are ordered by wealth if no key below a target's bin exceeds the target and none above it
        // falls short.  thr's neighbours must be strictly apart (the sums beside its bin were taken as > thr /
        // < thr) unless thr is a saturated value, whose copies beside its bin were counted apart.
        constexpr uint32_t KEY_ZERO = 0x80000000u, KEY_INF = 0xff800000u;
        const bool t_inf = thr_key == KEY_INF, t_zero = thr_key == KEY_ZERO;
        bool ok = true;
        for (int j = 0; j < 4; ++j)
          ok = ok && sh.ncand[rep[j]] <= CAND && sh.found[j] && sh.ext[j][0] <= sh.sel[j] && sh.sel[j] <= sh.ext[j][1];
        ok = ok && (t_inf || t_zero || (sh.ext[1][0] < thr_key && thr_key < sh.ext[1][1]));
        sh.lat_ok = ok;
        if (ok) {
          const long long fc_gt = (long long)f[2], fc_lt = (long long)f[3], fc_all = (long long)f[4];
          double coarse_gt = 0, coarse_lt = 0;
          long long cnt_gt = 0, sat[4] = {0, 0, 0, 0};   // +inf above, 0 above, +inf below, 0 below
          for (int q = 0; q < C; ++q) {
            coarse_gt += sh.part_d[q][0]; coarse_lt += sh.part_d[q][1];
            cnt_gt += sh.part_i[q][0];
            for (int u = 0; u < 4; ++u) sat[u] += sh.part_i[q][1 + u];
          }
          const double thr = (double)key_float(thr_key);
          const long long below = n - cnt_gt - sat[0] - sat[1] - fc_all;   // investors in the bins under thr's
          const long long n_gt = cnt_gt + (t_inf ? 0 : sat[0]) + (t_zero ? 0 : sat[1]) + fc_gt;
          const long long n_lt = below - (t_inf ? sat[2] : 0) - (t_zero ? sat[3] : 0) + fc_lt;
          if (!t_inf && sat[0] > 0) coarse_gt += INFINITY;
          const double sum_gt = fc_gt ? coarse_gt + f[0] : coarse_gt, sum_lt = fc_lt ? coarse_lt + f[1] : coarse_lt;
          const long long n_eq = n - n_gt - n_lt;
          const long long tt = K - n_gt;
          sh.res_i[6] = tt;
          sh.res_i[7] = n_eq - tt;
          sh.res_d[1] = (sum_gt + (tt > 0 ? (double)tt * thr : 0.0)) / (double)K;
          sh.res_d[2] = (sum_lt + (n_eq - tt > 0 ? (double)(n_eq - tt) * thr : 0.0)) / (double)(n - K);
        }
      }
    }
    cluster.sync();
    STAMP();
    radix = !L->lat_ok;
#pragma unroll
    for (int j = 0; j < 4; ++j) key_j[j] = L->sel[j];
  }

  if (radix) {
    if (r == 0 && tid == 0) atomicAdd(reinterpret_cast<unsigned long long*>(header + TH_RADIX), 1ull);
    // ---- pass 0: sum, count, level-1 histogram
    for (int i = tid; i < SL1; i += SEL_THREADS) sh.hist[i] = 0;
    cluster.sync();
    STAMP();
    {
      a0 = 0;
      c0 = 0;
      sweep([&](float x, uint32_t c, bool in) {
        a0 += (double)c * (double)x;      // c = 0 where the lane holds nothing
        c0 += c;
        warp_hist_add(sh.hist, float_key(x) >> 21, c, in);
      });
      STAMP();
      push_hist(sh.hist, L->hist, SL1, r);
      a0 = block_sum(a0, sh.red_d);
      c0 = block_sum(c0, sh.red_i);
      if (tid == 0) { L->part_d[r][0] = a0; L->part_i[r][0] = c0; }
    }
    cluster.sync();
    STAMP();
    if (r == 0) {
      if (tid == 0) {
        double sum_all = 0;
        long long cnt_all = 0;
        for (int q = 0; q < C; ++q) { sum_all += sh.part_d[q][0]; cnt_all += sh.part_i[q][0]; }
        if (cnt_all != n) header[TH_MISMATCH] = 1;
        // key bins that can only hold non-finite values: 3 = -inf, 2044 = +inf, 2047 = NaN
        const long long ninf = sh.hist[3], pinf = sh.hist[2044], nan = sh.hist[2047];
        const long long hi_ = pinf + nan;
        sh.res_i[0] = (hi_ + ninf) > 0; sh.res_i[1] = hi_ > 0 || ninf > n - K; sh.res_i[2] = hi_ > K || ninf > 0;
        sh.res_i[3] = nan > 0; sh.res_i[4] = nan > 0; sh.res_i[5] = nan > K;
        sh.res_d[0] = sum_all / (double)n;
      }
      scan_hists(sh.hist, SL1, 1, sh.warp_tot);   // (thread 0's reads above precede the scan's first barrier)
      if (tid < 4) {
        int bin; long long rem;
        find_rank(sh.hist, SL1, ranks[tid], bin, rem);
        sh.res_i[8 + tid] = bin; sh.res_i[12 + tid] = rem;
      }
    }
    cluster.sync();
    uint32_t pre[4];
    long long rk[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { pre[j] = (uint32_t)L->res_i[8 + j]; rk[j] = L->res_i[12 + j]; }
    STAMP();
    // targets that share a prefix share a histogram: only the first of them (its representative) is counted,
    // the leader copies it for the others before it scans
    int rep[4];
    auto find_reps = [&]() {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        rep[j] = j;
#pragma unroll
        for (int q = 3; q >= 0; --q)
          if (q < j && pre[q] == pre[j]) rep[j] = q;
      }
    };
    auto copy_reps = [&](int bins) {     // leader only
      for (int j = 1; j < 4; ++j)
        if (rep[j] != j)
          for (int i = tid; i < bins; i += SEL_THREADS) sh.hist[j * bins + i] = sh.hist[rep[j] * bins + i];
      __syncthreads();
    };
    find_reps();

    // ---- pass 1: level-2 histograms of the elements in the targets' level-1 bins
    // (the leader next writes its results after the barrier that ends the pass: every read above is done by then)
    for (int j = 0; j < 4; ++j)
      if (rep[j] == j)
        for (int i = tid; i < SL2; i += SEL_THREADS) sh.hist[j * SL2 + i] = 0;
    cluster.sync();
    {
      sweep([&](float x, uint32_t c, bool in) {
        const uint32_t k = float_key(x);
        const uint32_t b1 = k >> 21, b2 = (k >> 10) & (SL2 - 1);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (rep[j] == j) warp_hist_add(sh.hist + j * SL2, b2, c, in && b1 == pre[j]);     // (rep is warp-uniform)
      });
      STAMP();
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (rep[j] == j) push_hist(sh.hist + j * SL2, L->hist + j * SL2, SL2, r);
    }
    STAMP();
    cluster.sync();
    STAMP();
    if (r == 0) {
      copy_reps(SL2);
      scan_hists(sh.hist, SL2, 4, sh.warp_tot);
      if (tid < 4) {
        int bin; long long rem;
        find_rank(sh.hist + tid * SL2, SL2, rk[tid], bin, rem);
        sh.res_i[8 + tid] = bin; sh.res_i[12 + tid] = rem;
      }
    }
    cluster.sync();
#pragma unroll
    for (int j = 0; j < 4; ++j) { pre[j] = (pre[j] << 11) | (uint32_t)L->res_i[8 + j]; rk[j] = L->res_i[12 + j]; }   // 22 bits
    find_reps();
    STAMP();

    // ---- pass 2: level-3 histograms + the sums on either side of thr's 22-bit prefix
    for (int j = 0; j < 4; ++j)
      if (rep[j] == j)
        for (int i = tid; i < SL3; i += SEL_THREADS) sh.hist[j * SL3 + i] = 0;
    cluster.sync();
    const uint32_t thr22 = pre[1];
    {
      double v[2] = {0, 0};
      long long c_gt = 0;
      sweep([&](float x, uint32_t c, bool in) {
        const uint32_t k = float_key(x);
        const uint32_t hi22 = k >> 10;
        const double cx = (double)c * (double)x;
        if (in && hi22 > thr22) { v[0] += cx; c_gt += c; }
        else if (in && hi22 < thr22) v[1] += cx;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (rep[j] == j) warp_hist_add(sh.hist + j * SL3, k & (SL3 - 1), c, in && hi22 == pre[j]);
      });
      STAMP();
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (rep[j] == j) push_hist(sh.hist + j * SL3, L->hist + j * SL3, SL3, r);
      STAMP();
      block_sum_n<2>(v, sh.red_d2);
      c_gt = block_sum(c_gt, sh.red_i);
      if (tid == 0) { L->part_d[r][0] = v[0]; L->part_d[r][1] = v[1]; L->part_i[r][0] = c_gt; }
    }
    cluster.sync();
    if (r == 0) {
      // thr's level-3 histogram: bin `b3` holds the copies of the ONE fp32 value with key (prefix22 << 10 | b3).
      // The scan overwrites the counts with prefixes; the per-bin counts are read back as differences.
      copy_reps(SL3);
      scan_hists(sh.hist, SL3, 4, sh.warp_tot);
      if (tid < 4) {
        int bin; long long rem;
        find_rank(sh.hist + tid * SL3, SL3, rk[tid], bin, rem);
        sh.res_i[8 + tid] = bin; sh.res_i[12 + tid] = rem;
      }
      __syncthreads();
      const uint32_t thr_key = (pre[1] << 10) | (uint32_t)sh.res_i[8 + 1];
      const uint32_t thr_lo = thr_key & (SL3 - 1), base = thr_key & ~(uint32_t)(SL3 - 1);
      double f[5] = {0, 0, 0, 0, 0};      // sum > thr, sum < thr, count > thr, count < thr, count of the whole histogram
      const uint32_t* h3 = sh.hist + 1 * SL3;
      for (uint32_t b3 = tid; b3 < (uint32_t)SL3; b3 += SEL_THREADS) {
        const long long c = (long long)h3[b3] - (b3 > 0 ? (long long)h3[b3 - 1] : 0);
        f[4] += (double)c;                  // counts < 2^32: exact in fp64
        if (c == 0 || b3 == thr_lo) continue;   // an empty bin must not contribute 0 * inf
        const double val = (double)c * (double)key_float(base | b3);
        if (b3 > thr_lo) { f[0] += val; f[2] += (double)c; } else { f[1] += val; f[3] += (double)c; }
      }
      block_sum_n<5>(f, sh.red_d2);
      if (tid == 0) {
        const long long fc_gt = (long long)f[2], fc_lt = (long long)f[3], fc_all = (long long)f[4];
        double coarse_gt = 0, coarse_lt = 0;
        long long cnt_gt = 0;
        for (int q = 0; q < C; ++q) { coarse_gt += sh.part_d[q][0]; coarse_lt += sh.part_d[q][1]; cnt_gt += sh.part_i[q][0]; }
        const double thr = (double)key_float(thr_key);
        const long long n_gt = cnt_gt + fc_gt, n_lt = (n - cnt_gt - fc_all) + fc_lt;
        const double sum_gt = fc_gt ? coarse_gt + f[0] : coarse_gt, sum_lt = fc_lt ? coarse_lt + f[1] : coarse_lt;
        const long long n_eq = n - n_gt - n_lt;
        const long long tt = K - n_gt;   // ties that belong to the top group
        sh.res_i[6] = tt;
        sh.res_i[7] = n_eq - tt;
        sh.res_d[1] = (sum_gt + (tt > 0 ? (double)tt * thr : 0.0)) / (double)K;                       // mean_top
        sh.res_d[2] = (sum_lt + (n_eq - tt > 0 ? (double)(n_eq - tt) * thr : 0.0)) / (double)(n - K);   // mean_adj
      }
    }
    cluster.sync();
#pragma unroll
    for (int j = 0; j < 4; ++j) key_j[j] = (pre[j] << 10) | (uint32_t)L->res_i[8 + j];
    STAMP();
  }
  const uint32_t thr_key = key_j[1];
  const double mean_a = L->res_d[0], mean_t = L->res_d[1], mean_j = L->res_d[2];

  // ---- pass 3: deviations
  double d[6] = {0, 0, 0, 0, 0, 0};
  sweep([&](float x, uint32_t ci, bool in) {
    const double c = (double)ci;          // 0 where the lane holds nothing
    const uint32_t k = float_key(x);
    const double xd = (double)x;
    const double da = xd - mean_a;
    d[4] += c * fabs(da);
    d[5] += c * (da * da);
    if (k < thr_key) { const double e = xd - mean_j; d[2] += c * fabs(e); d[3] += c * (e * e); }
    else if (k > thr_key) { const double e = xd - mean_t; d[0] += c * fabs(e); d[1] += c * (e * e); }
  });
  STAMP();
  block_sum_n<6>(d, sh.red_d2);
  STAMP();
  if (tid == 0) {                        // (the leader consumed pass 2's partials before the last barrier)
#pragma unroll
    for (int q = 0; q < 6; ++q) L->part_d[r][q] = d[q];
  }
  cluster.sync();
  STAMP();
  if (r == 0 && tid == 0) {
    double d0 = 0, d1 = 0, d2 = 0, d3 = 0, d4 = 0, d5 = 0;
    for (int q = 0; q < C; ++q) {
      d0 += sh.part_d[q][0]; d1 += sh.part_d[q][1]; d2 += sh.part_d[q][2];
      d3 += sh.part_d[q][3]; d4 += sh.part_d[q][4]; d5 += sh.part_d[q][5];
    }
    const double thr = (double)key_float(thr_key);
    const double dt = thr - mean_t, da = thr - mean_j;
    const double tt = (double)sh.res_i[6], ta = (double)sh.res_i[7];
    // a tie share of zero must not contribute inf * 0
    const double abs_top = d0 + (tt > 0 ? tt * fabs(dt) : 0.0);
    const double sq_top = d1 + (tt > 0 ? tt * dt * dt : 0.0);
    const double abs_adj = d2 + (ta > 0 ? ta * fabs(da) : 0.0);
    const double sq_adj = d3 + (ta > 0 ? ta * da * da : 0.0);
    s[0] = mean_a; s[1] = mean_t; s[2] = mean_j;
    s[3] = d4 / (double)n; s[4] = abs_top / (double)K; s[5] = abs_adj / (double)(n - K);
    s[6] = sqrt(d5 / (double)n); s[7] = sqrt(sq_top / (double)K); s[8] = sqrt(sq_adj / (double)(n - K));
    s[9] = (double)key_float(key_j[0]); s[10] = (double)key_float(key_j[2]); s[11] = (double)key_float(key_j[3]);
    // torch semantics (see rowstats_resolve_kernel<3>): a non-finite member makes mean / std / MAD
    // nan, except that a one-element group's mean is the element itself; median propagates NaN
    const long long size[3] = {n, K, n - K};
    const double single[3] = {qnan, thr, (double)key_float(key_j[3])};
    for (int j = 0; j < 3; ++j) {
      if (sh.res_i[j]) { s[0 + j] = size[j] == 1 ? single[j] : qnan; s[3 + j] = qnan; s[6 + j] = qnan; }
      if (sh.res_i[3 + j]) s[9 + j] = qnan;
    }
  }
}

// Cluster size and per-CTA shared-memory cache of the select kernel.  Defaults from measurement on
// B200 (DESIGN.md): B200_SELECT_CLUSTER / B200_SELECT_CACHE override them for experiments.
static void select_shape(int& cluster, int& cache, bool early) {
  static int c = [] {
    const char* e = getenv("B200_SELECT_CLUSTER");
    if (e == nullptr) return 0;
    const int x = atoi(e);
    return x < 1 ? 1 : x > SEL_MAX_CLUSTER ? SEL_MAX_CLUSTER : x;
  }();
  static int k = [] {
    const char* e = getenv("B200_SELECT_CACHE");
    int x = e ? atoi(e) : 16384;
    return x < 0 ? 0 : x > 20480 ? 20480 : x;
  }();
  // 0: six CTAs per grid point, three when the select is launched early - the next sweep then has the other
  // 88 SMs (of 148) while the select runs, and 3 x 16 384 cached bins still hold the flagship's 45 561
  cluster = c != 0 ? c : early ? 3 : 6;
  cache = k;
}

template <int K>
static int launch_select_k(int n_grid, long long* header, const unsigned long long* ukeys, const uint32_t* ucnt,
                           float* wbuf, int64_t ldw, int32_t H, const LogTable& lf, double logV0, int64_t n_total,
                           int64_t top, double* stats, bool beside_sweep, bool force_radix, bool early,
                           cudaStream_t st) {
  static bool attr_set[64] = {false};
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  int C = 1, cache = 0;
  select_shape(C, cache, early);
  static const bool forced = getenv("B200_SELECT_CLUSTER") != nullptr;
  if (beside_sweep && !forced) C = 2;     // a small footprint beside a running sweep (B200_LEV_FLAG_BESIDE_SWEEP)
  const size_t dyn = (size_t)cache * 10;   // wealth, count and log-wealth bin of the cached bins
  if (dev < 64 && !attr_set[dev]) {
    B200_CUDA(cudaFuncSetAttribute(tally_select_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    if (C > 8) B200_CUDA(cudaFuncSetAttribute(tally_select_kernel<K>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    attr_set[dev] = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(n_grid * C));
  cfg.blockDim = dim3(SEL_THREADS);
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)C;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  set_pdl_attribute(at[1]);
  cfg.attrs = at;
  cfg.numAttrs = early ? 2 : 1;
  return check_cuda(cudaLaunchKernelEx(&cfg, tally_select_kernel<K>, header, ukeys, ucnt, wbuf, ldw, H, lf, logV0,
                                       n_total, top, stats, (int32_t)cache, (int32_t)force_radix),
                    "tally_select launch");
}

static int grid_for(int64_t work, int threads, int per_sm) {
  const int64_t want = (work + threads - 1) / threads;
  const int64_t cap = (int64_t)sm_count() * per_sm;
  return (int)std::max<int64_t>(1, std::min(want, cap));
}

}  // namespace b200

using namespace b200;

extern "C" int64_t b200_tally_workspace_bytes(const b200_tally_plan* plan) {
  if (plan_ok(plan)) return -1;
  return layout(*plan, nullptr).bytes;
}

extern "C" int64_t b200_tally_exchange_bytes(const b200_tally_plan* plan) {
  if (plan_ok(plan)) return -1;
  if (plan->world == 1) return 0;
  const TallyLayout L = layout(*plan, nullptr);
  return EX_FLAG_BYTES + 2 * ((exchange_list_bytes(L.list_cap) + 255) & ~(int64_t)255);
}

extern "C" int b200_tally_reset(const b200_tally_plan* plan, void* workspace, void* stream) {
  if (int rc = plan_ok(plan)) return rc;
  B200_REQUIRE(workspace != nullptr, "tally_reset: workspace is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  const TallyLayout L = layout(*plan, workspace);
  B200_CUDA(cudaMemsetAsync(L.header, 0, TH_WORDS * 8, st));
  tally_clear_kernel<<<grid_for((int64_t)L.capA, 256, 8), 256, 0, st>>>(L.keysA, L.countsA, nullptr, nullptr, L.capA);
  if (plan->world > 1)
    tally_clear_kernel<<<grid_for((int64_t)L.capB, 256, 8), 256, 0, st>>>(L.keysB, nullptr, L.countsB, L.posB, L.capB);
  return check_cuda(cudaGetLastError(), "tally_reset launch");
}

extern "C" int b200_tally_finalize(const b200_tally_plan* plan, void* workspace, const b200_tally_peers* peers,
                                   int32_t phase, void* stream) {
  if (int rc = plan_ok(plan)) return rc;
  B200_REQUIRE(workspace != nullptr, "tally_finalize: workspace is NULL");
  B200_REQUIRE(phase >= -1 && phase <= 1, "tally_finalize: phase must be -1, 0 or 1");
  cudaStream_t st = (cudaStream_t)stream;
  const TallyLayout L = layout(*plan, workspace);
  TallyDev t{L.keysA, L.countsA, L.header, L.capA - 1};
  PeerView P;
  memset(&P, 0, sizeof(P));
  const int cgrid = (int)((L.capA + COMPACT_CHUNK - 1) / COMPACT_CHUNK);
  if (plan->world == 1) {
    if (phase == 1) return 0;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)cgrid);
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    set_pdl_attribute(at[0]);
    cfg.attrs = at;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return check_cuda(cudaLaunchKernelEx(&cfg, tally_compact_kernel<false>, t, L.ukeys, L.ucnt,
                                         (int64_t)std::min(plan->bins_cap, L.list_cap), P),
                      "tally_compact launch");
  }
  B200_REQUIRE(peers != nullptr, "tally_finalize: peers is NULL with world > 1");
  B200_REQUIRE(peers->world == plan->world && peers->rank >= 0 && peers->rank < peers->world,
               "tally_finalize: peers->world / rank do not fit the plan");
  B200_REQUIRE(peers->epoch >= 1, "tally_finalize: epoch starts at 1");
  const int64_t lbytes = (exchange_list_bytes(L.list_cap) + 255) & ~(int64_t)255;
  P.world = peers->world; P.rank = peers->rank; P.epoch = peers->epoch;
  for (int r = 0; r < peers->world; ++r) {
    B200_REQUIRE(peers->exchange[r] != nullptr, "tally_finalize: exchange buffer of rank %d is NULL", r);
    char* ex = (char*)peers->exchange[r];
    char* lst = ex + EX_FLAG_BYTES + (peers->epoch & 1) * lbytes;
    P.flags[r] = (uint32_t*)ex;
    P.list_count[r] = (long long*)lst;
    P.list[r] = (BinEntry*)(lst + 16);
  }
  if (phase != 1) {
    tally_compact_kernel<true><<<cgrid, 256, 0, st>>>(t, nullptr, nullptr, L.list_cap, P);
    B200_CUDA(cudaGetLastError());
  }
  if (phase == 0) return 0;
  const int64_t cat = (int64_t)plan->world * L.list_cap;
  tally_merge_kernel<<<sm_count() * 2, 256, 0, st>>>(P, L.header, L.concat, L.slot_of, L.keysB, L.countsB, L.posB,
                                                     L.capB, cat);
  B200_CUDA(cudaGetLastError());
  const unsigned mgrid = (unsigned)std::min<int64_t>(L.nblk, (int64_t)sm_count() * 2);
  tally_mark_kernel<<<mgrid, 256, 0, st>>>(L.header, L.slot_of, L.posB, L.blockcnt);
  B200_CUDA(cudaGetLastError());
  tally_unique_kernel<<<mgrid, 256, 0, st>>>(L.header, L.concat, L.slot_of, L.keysB, L.countsB, L.posB,
                                                        L.blockcnt, L.ukeys, L.ucnt, plan->bins_cap);
  return check_cuda(cudaGetLastError(), "tally_unique launch");
}

extern "C" int b200_tally_stats(const b200_tally_plan* plan, void* workspace, const b200_lev_desc* desc,
                                const float* factors_host, int64_t n_total, int64_t top, double* stats, void* stream) {
  if (int rc = plan_ok(plan)) return rc;
  B200_REQUIRE(workspace != nullptr && desc != nullptr && factors_host != nullptr && stats != nullptr,
               "tally_stats: NULL argument");
  B200_REQUIRE(desc->n_grid >= 1 && desc->n_grid <= plan->grid_cap, "tally_stats: n_grid must be in 1..grid_cap");
  B200_REQUIRE(desc->n_outcomes >= 2 && desc->n_outcomes <= B200_MAX_OUTCOMES, "tally_stats: n_outcomes out of range");
  B200_REQUIRE(desc->horizon >= 1 && desc->horizon <= TALLY_MAX_HORIZON, "tally_stats: horizon out of range");
  B200_REQUIRE(n_total >= 2 && n_total < ((int64_t)1 << 32), "tally_stats: need 2 <= n_total < 2^32");
  B200_REQUIRE(top >= 1 && top < n_total, "tally_stats: need 1 <= top < n_total (top=%lld)", (long long)top);
  cudaStream_t st = (cudaStream_t)stream;
  const TallyLayout L = layout(*plan, workspace);
  LogTable lf;
  for (int k = 0; k < B200_MAX_OUTCOMES; ++k)
    for (int g = 0; g < B200_MAX_GRID; ++g) {
      double v = 0.0;
      if (g < desc->n_grid && k < desc->n_outcomes) {
        const float m = factors_host[(int64_t)g * desc->n_outcomes + k];
        if (m < 0.0f) return set_error(B200_EINVAL, "tally_stats: factors must be >= 0 (m[%d][%d] = %g)", g, k, (double)m);
        v = log((double)m);
      }
      lf.lm[k][g] = v;
    }
  const double logV0 = log((double)desc->value_0);
  const bool beside = (desc->flags & B200_LEV_FLAG_BESIDE_SWEEP) != 0;
  const bool radix = (desc->flags & B200_LEV_FLAG_RADIX_SELECT) != 0;
  // one GPU, nothing beside it: the select starts under the compaction, and the next sweep under the select
  const bool early = plan->world == 1 && !beside && pdl_enabled();
  switch (desc->n_outcomes) {
    case 2: return launch_select_k<2>(desc->n_grid, L.header, L.ukeys, L.ucnt, L.wbuf, L.ldw, desc->horizon, lf, logV0, n_total, top, stats, beside, radix, early, st);
    case 3: return launch_select_k<3>(desc->n_grid, L.header, L.ukeys, L.ucnt, L.wbuf, L.ldw, desc->horizon, lf, logV0, n_total, top, stats, beside, radix, early, st);
    default: return launch_select_k<4>(desc->n_grid, L.header, L.ukeys, L.ucnt, L.wbuf, L.ldw, desc->horizon, lf, logV0, n_total, top, stats, beside, radix, early, st);
  }
}
