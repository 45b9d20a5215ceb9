// Dense low-cardinality pass of a handle whose groups are known: sums only.
//
// A full dense pass (lowcard.cuh) finds, besides the sums, every group's row count and first row and ranks the groups
// by first row.  All of that depends on the keys alone, and a handle's keys do not change, so after one full dense pass
// of the narrow set whose clean status the host has read back (and whose value column had no validity bitmap, so that
// count = group size) the handle keeps those facts: k_lowcard_known_record copies them out of the GroupResult into
// handle-owned buffers.  Later narrow-set passes over value columns without a bitmap then run k_lowcard_sums:
//  * per warp: sum 8 B x GP and ONE TAG BYTE x GP instead of the 4-byte count word.  A lane claims its slot by storing
//    `lane | LK_SEEN` (STS.8) and reads the byte back (LDS.U8): per 32-row batch the count-word store goes and the
//    count-word load becomes a byte load whose slots share a bank word four to one.  Bit 7 stays set once a lane has
//    claimed the slot, which is what the full kernel's count word says when it is not CNT_UNSEEN.
//  * no first-row atomics and no rank kernel: k_lowcard_sums_merge writes each group's sum at its known rank and copies
//    the group's count, first row and key back into the GroupResult, so emit and everything after it see the state of
//    a full pass.
// The rows each warp reads, the duplicate folds (those of lc_accumulate), the warp / replica fold (skipping unseen
// slots) and the merge over CTAs (skipping CTAs that did not meet the id, lane-strided, same shuffle tree) are the full
// pass's at the same window, replication and grid: the sums are the full pass's bit for bit.
#pragma once
#include "lowcard.cuh"

namespace pa {

constexpr uint32_t LK_SEEN = 0x80u;        // tag byte: some lane of this warp has claimed the slot
constexpr uint32_t LK_NORANK = 0xFFFFFFFFu;
constexpr uint32_t LK_MODE = 6u;           // status[ST_MODE] of a sum-only pass (timing()["mode"] == "dense-known")

struct LkHead {                            // the recording pass's dense window and group count
  unsigned long long base;
  uint32_t window, rlog, ngroups, pad;
};

// Device view of a handle's facts: id space of the narrow set (LcCfg<*, false>::GP ids), by-rank arrays of G entries.
struct LkFacts {
  LkHead* head;
  uint32_t* id_rank;   // [GP] dense id -> rank, LK_NORANK for ids without rows
  uint32_t* count;     // by rank
  uint32_t* first;
  uint64_t* key;
  uint8_t* kind;
};

struct LkSmem {
  static constexpr size_t GP = LcCfg<VC_F, false>::GP;
  static constexpr int WARPS = LcCfg<VC_F, false>::WARPS;
  static constexpr size_t OFF_MISC = 0;                        // 4 x u32 (LcCtx::misc)
  static constexpr size_t OFF_ACC = 16;
  static constexpr size_t W_SUM = 0;                           // GP x 8 B
  static constexpr size_t W_TAG = GP * 8;                      // GP x 1 B
  static constexpr size_t ACC_PER_WARP = ((W_TAG + GP + 15) / 16) * 16;
  static constexpr size_t TOTAL = OFF_ACC + ACC_PER_WARP * WARPS;
  static_assert(TOTAL <= 227 * 1024, "shared-memory layout exceeds 227 KB");
  static_assert(W_TAG % 4 == 0 && W_TAG + ((GP + 3) / 4) * 4 <= ACC_PER_WARP, "tag words are cleared as whole words");
};

__device__ __forceinline__ uint32_t lds8(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}

// the sum of lane `src` (the count and first row are known, so only the sum travels on the inline paths)
template <int VC>
__device__ __forceinline__ LcContrib<false> lk_pull(const LcContrib<false>& k, int src) {
  LcContrib<false> o = k;
  o.sum = __shfl_sync(0xFFFFFFFFu, k.sum, src);
  return o;
}

// lc_accumulate of the narrow dense set without count word and first row: `c.cw` is this warp's tag-byte array.
template <int VC, bool CLEAN>
__device__ __forceinline__ void lk_accumulate(uint32_t id, uint64_t vbits, bool vvalid, const LcCtx& c) {
  constexpr uint32_t FULL = 0xFFFFFFFFu;
  const uint32_t lane = lane_id();
  const bool live = CLEAN ? true : id != LC_NOID;
  const uint32_t ida = live ? id : 0u;
  const uint32_t tag_addr = c.cw + ida, sum_addr = c.sum + ida * 8u;
  const bool vv = CLEAN ? true : vvalid;
  LcContrib<false> k;
  k.sum = vv ? vbits : 0ull;
  k.cnt = 0u;
  k.lo = lane;
  if (live) sts8(tag_addr, lane | LK_SEEN);
  __syncwarp();
  const uint32_t tb = lds8(tag_addr);
  uint64_t s = lds64(sum_addr);
  const uint32_t tag = tb & 31u;
  const bool winner = live && (tb == (lane | LK_SEEN));
  const uint32_t losers = __ballot_sync(FULL, live && !winner);
  k.doer = winner;
  if (losers) {
    if ((losers & (losers - 1u)) == 0u) {
      const int L = __ffs(losers) - 1;
      const uint32_t tw = __shfl_sync(FULL, tag, L);
      const LcContrib<false> o = lk_pull<VC>(k, L);
      if (lane == tw) lc_add<VC, false>(k, o);
    } else {
      bool independent = false;
      int l0 = 0, l1 = 0, l2 = -1;
      uint32_t t0 = 0, t1 = 0, t2 = 0xFFFFFFFFu;
      if (__popc(losers) <= 3) {
        l0 = __ffs(losers) - 1;
        const uint32_t rest = losers & (losers - 1u);
        l1 = __ffs(rest) - 1;
        const uint32_t rest2 = rest & (rest - 1u);
        t0 = __shfl_sync(FULL, tag, l0);
        t1 = __shfl_sync(FULL, tag, l1);
        independent = t0 != t1;
        if (rest2) {
          l2 = __ffs(rest2) - 1;
          t2 = __shfl_sync(FULL, tag, l2);
          independent = independent && t2 != t0 && t2 != t1;
        }
      }
      if (independent) {
        const LcContrib<false> o0 = lk_pull<VC>(k, l0);
        const LcContrib<false> o1 = lk_pull<VC>(k, l1);
        if (lane == t0) lc_add<VC, false>(k, o0);
        if (lane == t1) lc_add<VC, false>(k, o1);
        if (l2 >= 0) {
          const LcContrib<false> o2 = lk_pull<VC>(k, l2);
          if (lane == t2) lc_add<VC, false>(k, o2);
        }
      } else {
        k = lc_fold_general<VC, false>(k, id, tag, live, losers);
      }
    }
  }
  if (k.doer) {
    if constexpr (VC == VC_F) {
      s = static_cast<uint64_t>(__double_as_longlong(__longlong_as_double(static_cast<long long>(s)) +
                                                     __longlong_as_double(static_cast<long long>(k.sum))));
    } else {
      s += k.sum;
    }
    sts64(sum_addr, s);
  }
  __syncwarp();
}

template <int VC, bool CLEAN>
__device__ __forceinline__ bool lk_process_group(const LcBuf& b, uint32_t lane, const LcCtx& c, const LcArgs& a) {
  uint32_t id[LC_NB];
  if (!lc_resolve_group<VC, false, true, CLEAN>(b, id, lane, c, a)) return false;
#pragma unroll
  for (int e = 0; e < LC_NB; ++e) {
    const bool vvalid = CLEAN ? true : ((b.vv >> e) & 1u) != 0;
    lk_accumulate<VC, CLEAN>(id[e], b.val[e], vvalid && (CLEAN || id[e] != LC_NOID), c);
  }
  return true;
}

// lc_scan_rows of the dense kernel: the same row groups per warp, in the same order.
template <int VC, bool FAST>
__device__ __forceinline__ void lk_scan_rows(const LcArgs& a, const LcCtx& c, int warp, uint32_t lane) {
  if (warp >= c.nwarps) return;
  const int64_t gw = static_cast<int64_t>(blockIdx.x) * c.nwarps + warp;
  const int64_t nw = static_cast<int64_t>(gridDim.x) * c.nwarps;
  const int64_t n_full = a.n / LC_GROUP_ROWS;
  const int64_t n_groups = (a.n + LC_GROUP_ROWS - 1) / LC_GROUP_ROWS;
  volatile uint32_t* abort_local = c.misc + 1;
  volatile uint32_t* abort_global = a.status + ST_ABORT;
  if constexpr (FAST) {
    LcBuf cur, nxt;
    int64_t g = gw;
    if (g < n_full) lc_load_fast(cur, a, g * LC_GROUP_ROWS, lane);
    while (g < n_full) {
      const int64_t gn = g + nw;
      const uint32_t gabort = *abort_global;
      if (gn < n_full) lc_load_fast(nxt, a, gn * LC_GROUP_ROWS, lane);
      if (!lk_process_group<VC, true>(cur, lane, c, a)) return;
      if (__any_sync(0xFFFFFFFFu, (*abort_local | gabort) != 0)) return;
      cur = nxt;
      g = gn;
    }
    if (n_groups > n_full && gw == (n_full % nw)) {
      LcBuf t;
      lc_load_generic<VC>(t, a, n_full * LC_GROUP_ROWS, lane);
      lk_process_group<VC, false>(t, lane, c, a);
    }
  } else {
    LcBuf cur, nxt;
    int64_t g = gw;
    if (g < n_groups) lc_load_generic<VC>(cur, a, g * LC_GROUP_ROWS, lane);
    while (g < n_groups) {
      const int64_t gn = g + nw;
      if (gn < n_groups) lc_load_generic<VC>(nxt, a, gn * LC_GROUP_ROWS, lane);
      const uint32_t gabort = *abort_global;
      if (!lk_process_group<VC, false>(cur, lane, c, a)) return;
      if (__any_sync(0xFFFFFFFFu, (*abort_local | gabort) != 0)) return;
      cur = nxt;
      g = gn;
    }
  }
}

// Sum-only dense scan.  Writes this CTA's partial sums to a.p_sum and, in a.p_count, 1 where the CTA met the id (the
// full pass's p_first != kNoRow) and 0 elsewhere.  A key outside the recorded window aborts with ST_DENSE_MISS.
template <int VC, bool FAST>
__global__ void __launch_bounds__(LkSmem::WARPS * 32, 1) k_lowcard_sums(LcArgs a, const LkHead* h) {
  using Cfg = LcCfg<VC, false>;
  using L = LkSmem;
  constexpr int THREADS = L::WARPS * 32;
  extern __shared__ __align__(16) unsigned char smem[];
  const int warp = threadIdx.x >> 5;
  const uint32_t lane = lane_id();
  LcCtx c{};
  c.misc = reinterpret_cast<uint32_t*>(smem + L::OFF_MISC);
  c.base = h->base;
  c.window = h->window;
  c.rlog = h->rlog;
  c.rmask = (1u << c.rlog) - 1u;
  const int nwarps = c.rlog >= 5 ? 12 : L::WARPS;   // k_lowcard_scan's choice for the narrow set: the same rows per warp
  c.nwarps = nwarps;
  unsigned char* my_acc = smem + L::OFF_ACC + L::ACC_PER_WARP * (warp < nwarps ? warp : 0);
  c.sum = smem_u32(my_acc) + static_cast<uint32_t>(L::W_SUM);
  c.cw = smem_u32(my_acc) + static_cast<uint32_t>(L::W_TAG);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    a.status[ST_MODE] = LK_MODE;
    a.status[ST_RLOG] = c.rlog;
  }
  if (threadIdx.x < 4) c.misc[threadIdx.x] = 0;
  if (warp < nwarps) {
    for (int i = lane; i < static_cast<int>(L::GP); i += 32) reinterpret_cast<uint64_t*>(my_acc + L::W_SUM)[i] = 0ull;
    for (int i = lane; i < static_cast<int>((L::GP + 3) / 4); i += 32) reinterpret_cast<uint32_t*>(my_acc + L::W_TAG)[i] = 0u;
  }
  __syncthreads();

  lk_scan_rows<VC, FAST>(a, c, warp, lane);
  __syncthreads();
  if (c.misc[1]) {
    if (threadIdx.x == 0) atomicExch(a.status + ST_ABORT, 1u);
    return;
  }

  // fold the warps and replicas in k_lowcard_scan's order, skipping the slots a warp never claimed
  const size_t pbase = static_cast<size_t>(blockIdx.x) * Cfg::GP;
  const uint32_t nrep = 1u << c.rlog;
  for (int id = threadIdx.x; id < Cfg::GP; id += THREADS) {
    const bool regular = id < Cfg::GMAX;
    const uint32_t reps = regular ? nrep : 1u;
    uint64_t sum = 0;
    double fsum = 0.0;
    uint32_t seen = 0;
    if (!regular || static_cast<uint32_t>(id) < c.window) {
      for (int w = 0; w < nwarps; ++w) {
        const unsigned char* wa = smem + L::OFF_ACC + L::ACC_PER_WARP * w;
        for (uint32_t r = 0; r < reps; ++r) {
          const uint32_t slot = regular ? ((static_cast<uint32_t>(id) << c.rlog) | r) : static_cast<uint32_t>(id);
          if (!(wa[L::W_TAG + slot] & LK_SEEN)) continue;
          seen = 1;
          const uint64_t s = reinterpret_cast<const uint64_t*>(wa + L::W_SUM)[slot];
          if constexpr (VC == VC_F) fsum += __longlong_as_double(static_cast<long long>(s));
          else sum += s;
        }
      }
    }
    if constexpr (VC == VC_F) sum = static_cast<uint64_t>(__double_as_longlong(fsum));
    a.p_sum[pbase + id] = sum;
    a.p_count[pbase + id] = seen;
  }
}

// One warp per id folds the CTAs that met it (k_lowcard_merge's order) and writes the group's sum at its known rank,
// with its count, first row and key from the facts.  An id the recording pass did not have aborts with ST_DENSE_MISS:
// the keys are not the ones the facts describe, and the full pass redoes the aggregate.
template <int VC>
__global__ void __launch_bounds__(256) k_lowcard_sums_merge(LmArgs a, LkFacts f) {
  using Cfg = LcCfg<VC, false>;
  constexpr uint32_t FULL = 0xFFFFFFFFu;
  const int id = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (id >= Cfg::GP) return;
  if (*reinterpret_cast<volatile uint32_t*>(a.status + ST_ABORT)) return;
  const uint32_t lane = lane_id();
  uint64_t sum = 0;
  double fsum = 0.0;
  bool seen = false;
  for (int b = lane; b < a.grid; b += 32) {
    const size_t p = static_cast<size_t>(b) * Cfg::GP + id;
    if (!a.part.p_count[p]) continue;
    seen = true;
    if constexpr (VC == VC_F) fsum += __longlong_as_double(static_cast<long long>(a.part.p_sum[p]));
    else sum += a.part.p_sum[p];
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    if constexpr (VC == VC_F) fsum += __shfl_xor_sync(FULL, fsum, d);
    else sum += __shfl_xor_sync(FULL, sum, d);
  }
  if (!__any_sync(FULL, seen) || lane != 0) return;
  const uint32_t r = f.id_rank[id];
  if (r == LK_NORANK) {
    atomicExch(a.status + ST_DENSE_MISS, 1u);
    atomicExch(a.status + ST_ABORT, 1u);
    return;
  }
  if constexpr (VC == VC_F) sum = static_cast<uint64_t>(__double_as_longlong(fsum));
  a.out.sum[r] = sum;
  a.out.count[r] = f.count[r];
  a.out.first_row[r] = f.first[r];
  a.out.key[r] = f.key[r];
  a.out.key_kind[r] = f.kind[r];
  atomicAdd(a.status + ST_NGROUPS, 1u);
}

// After k_lowcard_rank of a full narrow-set pass: copies the dense window, the group count, id -> rank and count /
// first row / key by rank into the handle's facts.  One CTA.  Nothing is written when the pass aborted or ran in hash
// mode; the host trusts the facts only once it has read back a clean dense status of this pass.
constexpr int LK_REC_THREADS = 256;
__global__ void __launch_bounds__(LK_REC_THREADS) k_lowcard_known_record(LmArgs a, LkFacts f) {
  using Cfg = LcCfg<VC_F, false>;
  const volatile uint32_t* st = a.status;
  if (st[ST_ABORT] || st[ST_MODE] != 1u) return;
  uint64_t base;
  uint32_t window, rlog;
  lc_dense_mode(a.part.dir.prep, 0, Cfg::GMAX, &base, &window, &rlog);
  for (int i = threadIdx.x; i < Cfg::GP; i += LK_REC_THREADS) f.id_rank[i] = LK_NORANK;
  __syncthreads();
  const uint32_t G = st[ST_NGROUPS];
  for (uint32_t r = threadIdx.x; r < G; r += LK_REC_THREADS) {
    const uint8_t kind = a.out.key_kind[r];
    const uint64_t key = a.out.key[r];
    const uint32_t id = kind == KK_NULL ? static_cast<uint32_t>(Cfg::ID_NULL) : static_cast<uint32_t>(key - base);
    if (id < static_cast<uint32_t>(Cfg::GP)) f.id_rank[id] = r;
    f.count[r] = a.out.count[r];
    f.first[r] = a.out.first_row[r];
    f.key[r] = key;
    f.kind[r] = kind;
  }
  if (threadIdx.x == 0) {
    f.head->base = base;
    f.head->window = window;
    f.head->rlog = rlog;
    f.head->ngroups = G;
  }
}

}  // namespace pa
