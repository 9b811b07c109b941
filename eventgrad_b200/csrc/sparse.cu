// eventgrad_b200 -- sparse (top-k) event exchange (K3) for sm_100a.
//
// spevent semantics (/root/reference/dcifar10/spevent/spevent.cpp:342-448): when tensor i
// fires, the k_i elements with the largest |theta - prev| travel as (value, index) pairs; the
// sender then sets prev[idx] = value; the receiver scatters the record into a persistent
// replica of that neighbour and mixes with the FULL replicas.
//
// Device design, round 2: THREE launches, three streaming passes over (theta, prev), for ALL fired tensors of
// the model at once (segmented by tensor: a tile belongs to exactly one tensor), nothing sorted, no host round
// trip.  (Round 1 needed 9 launches / 5 passes and was as slow as the dense step it is meant to undercut.)
//   1. sparse_hist_kernel   pass 1: shared-memory histogram of bits [30:20] of the monotone uint32 image of
//                           |diff|, merged per tensor; the CTA that completes a tensor picks the bucket that
//                           holds the k-th largest key (no separate scan launch).
//   2. sparse_cand_kernel   pass 2: the low 20 bits of every key in that bucket go to a compact per-tensor
//                           candidate list (one atomic per TILE, block-scan inside); the CTA that completes a
//                           tensor resolves the remaining 20 bits (11 + 9) on that small list alone ->
//                           exact threshold tau and the number of tau-ties to take.
//   3. sparse_compact_kernel pass 3: compaction straight into BOTH neighbours' record inboxes over NVLink + prev
//                           update: keys > tau take slots from one atomic per tile; ties at tau are resolved towards
//                           the lowest index (the selected SET is deterministic) by a look-back over per-tile tie
//                           counts that only tiles containing a tie perform.
// The receive side (scatter of freshly arrived records into the replicas) is the PROLOGUE of the dense
// mix+SGD kernel (gossip.cu, `sparse_apply_prologue` below + one grid barrier), so a spevent step is 4 launches.
#include "sparse_apply.cuh"

namespace egb {

// Radix digits of the key.  Keys are |x| bit patterns, so bit 31 is always 0: the first digit is bits [30:20]
// (8 exponent + 3 mantissa bits -- one bit finer than [31:21], which halves the candidate bucket), the second
// [19:9], the third [8:0].
#define SP_SH1 20
#define SP_SH2 9
__device__ __forceinline__ uint32_t diff_key(float a, float b) {
  return __float_as_uint(fabsf(__fsub_rn(a, b)));   // non-negative floats order like uints
}

// number of valid (non-padding) elements of tile t
__device__ __forceinline__ int tile_valid(const TableDev& tab, int t, int i) {
  const int first = (t - tab.t_tile_start[i]) * EG_TILE;
  const int rem = tab.t_numel[i] - first;
  return rem < EG_TILE ? rem : EG_TILE;
}

// Walk a shared-memory histogram of `nb` buckets (nb <= 2048, 256 threads x 8 buckets) from the TOP bucket down
// to the one holding the element of rank `remain` (1-based, counted from the largest).  Returns, to every thread,
// {bucket, number of elements in higher buckets}.  `sh` is left untouched.
__device__ __forceinline__ void block_pick(const unsigned int* sh, int nb, unsigned remain, unsigned* digit,
                                           unsigned* above) {
  __shared__ unsigned int wsum[EG_WARPS];
  __shared__ unsigned int s_digit, s_above;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned int loc[8], tot = 0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {                 // descending order: position q <-> bucket nb-1-q
    const int q = tid * 8 + e;
    const unsigned c = (q < nb) ? sh[nb - 1 - q] : 0u;
    loc[e] = c;
    tot += c;
  }
  unsigned int inc = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  __syncthreads();                               // previous use of wsum / s_digit is over
  if (lane == 31) wsum[warp] = inc;
  if (tid == 0) {
    s_digit = 0u;
    s_above = 0u;
  }
  __syncthreads();
  unsigned int woff = 0;
  for (int w = 0; w < warp; ++w) woff += wsum[w];
  unsigned int excl = woff + inc - tot;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    if (remain > excl && remain <= excl + loc[e]) {       // exactly one (thread, e) satisfies this
      s_digit = (unsigned)(nb - 1 - (tid * 8 + e));
      s_above = excl;
    }
    excl += loc[e];
  }
  __syncthreads();
  *digit = s_digit;
  *above = s_above;
}

// "Which tensors did this CTA complete?"  Tiles [t0, t1) were processed by this CTA; add the number of tiles it
// contributed to each tensor's completion counter; tensors whose counter reaches their tile count are returned
// in s_own (their data from EVERY CTA is visible after the fences).  Tiles ascend => equal tensors consecutive.
#define SP_MAX_OWN 64
__device__ __forceinline__ int claim_completed(const TableDev& tab, unsigned int* done, int t0, int t1, int* s_own,
                                               int* s_nown) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    int nown = 0, cur = -1, cnt = 0;
    for (int t = t0; t <= t1; ++t) {
      const int i = (t < t1) ? tab.tile_tensor[t] : -2;
      if (i != cur) {
        if (cur >= 0) {
          const unsigned prev = atomicAdd(done + cur, (unsigned)cnt);
          if (prev + (unsigned)cnt == (unsigned)tab.t_tile_count[cur]) {
            done[cur] = 0u;                                  // ready for the next step
            if (nown < SP_MAX_OWN) s_own[nown++] = cur;
          }
        }
        cur = i;
        cnt = 0;
      }
      ++cnt;
    }
    *s_nown = nown;
    __threadfence();
  }
  __syncthreads();
  return *s_nown;
}

// ---------------------------------------------------------------- 1. histogram of the top 11 key bits
__global__ void __launch_bounds__(EG_THREADS, 4) sparse_hist_kernel(const SparseParams p) {
  __shared__ unsigned int sh[SP_BINS];
  __shared__ int s_own[SP_MAX_OWN];
  __shared__ int s_nown;
  const int tid = threadIdx.x;
  const int G = gridDim.x;
  int per = (p.tab.n_tiles + G - 1) / G;                // blocked tile ranges: few tensor switches per CTA
  if (per > SP_MAX_OWN) per = SP_MAX_OWN;               // (host sizes the grid so that this never truncates)
  const int t0 = min(p.tab.n_tiles, blockIdx.x * per), t1 = min(p.tab.n_tiles, t0 + per);
  int cur = -1;
  auto flush = [&](int tensor) {
    __syncthreads();
    if (tensor >= 0) {
      for (int bkt = tid; bkt < SP_BINS; bkt += EG_THREADS) {
        const unsigned c = sh[bkt];
        if (c) atomicAdd(p.hist + (size_t)tensor * SP_BINS + bkt, c);
      }
    }
    for (int bkt = tid; bkt < SP_BINS; bkt += EG_THREADS) sh[bkt] = 0u;
    __syncthreads();
  };
  flush(-1);
  // software pipeline: the loads of tile t+1 are in flight while the shared-memory atomics of tile t execute
  F8 a, b, an, bn;
  auto fetch = [&](int t, F8& x, F8& y) {
    if (t < t1 && p.fire[p.tab.tile_tensor[t]]) {
      const size_t base = (size_t)t * EG_TILE + (size_t)tid * EG_VEC;
      x = ld_f8(p.theta + base);
      y = ld_f8(p.prev + base);
    }
  };
  fetch(t0, an, bn);
  for (int t = t0; t < t1; ++t) {
    a = an;
    b = bn;
    fetch(t + 1, an, bn);
    const int i = p.tab.tile_tensor[t];
    if (tid == 0) p.desc[t] = 0ull;                      // look-back descriptors of pass 3 start EMPTY
    if (!p.fire[i]) continue;
    if (i != cur) {
      flush(cur);
      cur = i;
    }
    const int valid = tile_valid(p.tab, t, i);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      if (tid * EG_VEC + e >= valid) continue;
      atomicAdd(&sh[diff_key(a.v[e], b.v[e]) >> SP_SH1], 1u);
    }
  }
  flush(cur);
  // ---- tensors completed by this CTA: pick the bucket of the k-th largest key, clear the histogram ----------
  const int nown = claim_completed(p.tab, p.done1, t0, t1, s_own, &s_nown);
  for (int o = 0; o < nown; ++o) {
    const int i = s_own[o];
    if (!p.fire[i]) continue;                            // uniform per CTA
    unsigned int* h = p.hist + (size_t)i * SP_BINS;
    __syncthreads();
    for (int bkt = tid; bkt < SP_BINS; bkt += EG_THREADS) {
      sh[bkt] = __ldcg(h + bkt);
      h[bkt] = 0u;                                       // ready for the next step
    }
    __syncthreads();
    unsigned digit, above;
    block_pick(sh, SP_BINS, (unsigned)p.t_k[i], &digit, &above);
    if (tid == 0) {
      p.sel_prefix[i] = digit;                           // bits [30:20] of tau
      p.sel_remain[i] = (unsigned)p.t_k[i] - above;      // rank inside that bucket
      p.cand_cnt[i] = 0u;
    }
  }
}

// ---------------------------------------------------------------- 2. candidates of the chosen bucket
__global__ void __launch_bounds__(EG_THREADS, 4) sparse_cand_kernel(const SparseParams p) {
  __shared__ unsigned int sh[SP_BINS];
  __shared__ unsigned int wsum[EG_WARPS];
  __shared__ unsigned int s_base;
  __shared__ int s_own[SP_MAX_OWN];
  __shared__ int s_nown;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x;
  int per = (p.tab.n_tiles + G - 1) / G;
  if (per > SP_MAX_OWN) per = SP_MAX_OWN;
  const int t0 = min(p.tab.n_tiles, blockIdx.x * per), t1 = min(p.tab.n_tiles, t0 + per);
  F8 a, b, an, bn;
  auto fetch = [&](int t, F8& x, F8& y) {
    if (t < t1 && p.fire[p.tab.tile_tensor[t]]) {
      const size_t base = (size_t)t * EG_TILE + (size_t)tid * EG_VEC;
      x = ld_f8(p.theta + base);
      y = ld_f8(p.prev + base);
    }
  };
  fetch(t0, an, bn);
  for (int t = t0; t < t1; ++t) {
    a = an;
    b = bn;
    fetch(t + 1, an, bn);                                 // next tile's loads overlap this tile's scan + atomic
    const int i = p.tab.tile_tensor[t];
    if (!p.fire[i]) continue;
    const uint32_t prefix = p.sel_prefix[i];
    const int valid = tile_valid(p.tab, t, i);
    uint32_t keys[8];
    unsigned m = 0, c = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      keys[e] = diff_key(a.v[e], b.v[e]);
      if (tid * EG_VEC + e < valid && (keys[e] >> SP_SH1) == prefix) {
        m |= 1u << e;
        ++c;
      }
    }
    // block exclusive scan of c; ONE global atomic per tile reserves the tile's slice of the candidate list
    unsigned inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += v;
    }
    __syncthreads();
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    unsigned woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < EG_WARPS; ++w) {
      if (w < warp) woff += wsum[w];
      total += wsum[w];
    }
    if (tid == 0) s_base = total ? atomicAdd(p.cand_cnt + i, total) : 0u;
    __syncthreads();
    if (c) {
      uint32_t* dst = p.cand + (size_t)p.tab.t_tile_start[i] * EG_TILE + s_base + woff + inc - c;
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (m & (1u << e)) *dst++ = keys[e] & ((1u << SP_SH1) - 1u);
    }
  }
  // ---- tensors completed by this CTA: resolve the remaining 20 bits on the candidate list alone --------------
  const int nown = claim_completed(p.tab, p.done2, t0, t1, s_own, &s_nown);
  for (int o = 0; o < nown; ++o) {
    const int i = s_own[o];
    if (!p.fire[i]) continue;
    const uint32_t* cand = p.cand + (size_t)p.tab.t_tile_start[i] * EG_TILE;
    const unsigned n = __ldcg(p.cand_cnt + i);
    unsigned remain = p.sel_remain[i];
    // digit 2: bits [19:9]
    __syncthreads();
    for (int bkt = tid; bkt < SP_BINS; bkt += EG_THREADS) sh[bkt] = 0u;
    __syncthreads();
    for (unsigned j0 = 0; j0 < n; j0 += 8 * EG_THREADS) {           // 8 independent L2 loads in flight per thread
      uint32_t cv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const unsigned j = j0 + u * EG_THREADS + tid;
        cv[u] = (j < n) ? __ldcg(cand + j) : 0xFFFFFFFFu;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (cv[u] != 0xFFFFFFFFu) atomicAdd(&sh[cv[u] >> SP_SH2], 1u);
    }
    __syncthreads();
    unsigned d2, above;
    block_pick(sh, SP_BINS, remain, &d2, &above);
    remain -= above;
    // digit 3: bits [8:0] among the candidates that match digit 2
    __syncthreads();
    for (int bkt = tid; bkt < (1 << SP_SH2); bkt += EG_THREADS) sh[bkt] = 0u;
    __syncthreads();
    for (unsigned j0 = 0; j0 < n; j0 += 8 * EG_THREADS) {
      uint32_t cv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const unsigned j = j0 + u * EG_THREADS + tid;
        cv[u] = (j < n) ? __ldcg(cand + j) : 0xFFFFFFFFu;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (cv[u] != 0xFFFFFFFFu && (cv[u] >> SP_SH2) == d2) atomicAdd(&sh[cv[u] & ((1u << SP_SH2) - 1u)], 1u);
    }
    __syncthreads();
    unsigned d3;
    block_pick(sh, 1 << SP_SH2, remain, &d3, &above);
    if (tid == 0) {
      p.sel_prefix[i] = (p.sel_prefix[i] << SP_SH1) | (d2 << SP_SH2) | d3;    // tau: the k-th largest key, exactly
      p.sel_remain[i] = remain - above;                               // how many keys == tau are selected (>= 1)
      p.cand_cnt[i] = 0u;                                             // pass 3 reuses it as the slot counter of keys > tau
    }
  }
}

// ---------------------------------------------------------------- 3. compaction -> peers
// Slots of a tensor's record: [0, need_eq) the selected ties (keys == tau; the need_eq LOWEST indices win, so the
// selected set is deterministic), then every key > tau.  Keys > tau take their slots from one atomic reservation per
// tile (their order inside the record is irrelevant: the receiver scatters by index).  Ties are ordered by a
// look-back over per-tile tie counts, performed only by tiles that contain a tie and cut short as soon as need_eq
// earlier ties have been seen -- in the common case (one element equals tau) a single tile per tensor looks back.
// Descriptor of a tile: [63:62] = 1 once published, [31:0] number of keys == tau in the tile.
#define SP_AGG (1ull << 62)
__device__ __forceinline__ unsigned long long ld_desc(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_desc(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(EG_THREADS, 4) sparse_compact_kernel(const SparseParams p) {
  __shared__ unsigned int wg[EG_WARPS], we[EG_WARPS];
  __shared__ unsigned int s_gbase, s_pe;                // slot base of this tile's keys > tau; ties before this tile
  __shared__ int s_last, s_ok;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int step = *p.pass_num + 1;
  const int G = gridDim.x;
  if (p.sync) {
    if (tid == 0) {   // WAR guard on the neighbours' record inboxes
      bool ok = wait_ge(p.ack_from_l, (uint32_t)(step - 1), p.status, p.timeout_ns);
      ok = wait_ge(p.ack_from_r, (uint32_t)(step - 1), p.status, p.timeout_ns) && ok;
      s_ok = ok ? 1 : 0;
    }
    __syncthreads();
    if (!s_ok) return;                                  // wedged peer: store nothing (status is sticky)
  }
  // tiles in ASCENDING order, strided over the persistent (co-resident) grid: a tile that has to look back only
  // waits for tiles that are already being processed
  F8 a, b, an, bn;
  auto fetch = [&](int t, F8& x, F8& y) {
    if (t < p.tab.n_tiles && p.fire[p.tab.tile_tensor[t]]) {
      const size_t base = (size_t)t * EG_TILE + (size_t)tid * EG_VEC;
      x = ld_f8(p.theta + base);
      y = ld_f8(p.prev + base);
    }
  };
  fetch(blockIdx.x, an, bn);
  for (int t = blockIdx.x; t < p.tab.n_tiles; t += G) {
    a = an;
    b = bn;
    fetch(t + G, an, bn);                               // next tile's loads overlap this tile's scan / atomics
    const int i = p.tab.tile_tensor[t];
    if (!p.fire[i]) continue;
    const uint32_t tau = p.sel_prefix[i];
    const unsigned need_eq = p.sel_remain[i];
    const int k = p.t_k[i];
    const int ts = p.tab.t_tile_start[i];
    const int valid = tile_valid(p.tab, t, i);
    const int first = (t - ts) * EG_TILE;
    const size_t base = (size_t)t * EG_TILE + (size_t)tid * EG_VEC;
    unsigned fg = 0, fe = 0, g = 0, q = 0;   // bit masks + counts
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      if (tid * EG_VEC + e >= valid) continue;
      const uint32_t key = diff_key(a.v[e], b.v[e]);
      if (key > tau) {
        fg |= 1u << e;
        ++g;
      } else if (key == tau) {
        fe |= 1u << e;
        ++q;
      }
    }
    unsigned gi = g, qi = q;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned vg = __shfl_up_sync(0xffffffffu, gi, o), vq = __shfl_up_sync(0xffffffffu, qi, o);
      if (lane >= o) {
        gi += vg;
        qi += vq;
      }
    }
    __syncthreads();                                    // previous tile's readers of wg / s_gbase are done
    if (lane == 31) {
      wg[warp] = gi;
      we[warp] = qi;
    }
    __syncthreads();
    if (warp == 0) {
      unsigned G2 = 0, Q2 = 0;
#pragma unroll
      for (int w = 0; w < EG_WARPS; ++w) {
        G2 += wg[w];
        Q2 += we[w];
      }
      if (lane == 0) {
        st_desc(p.desc + t, SP_AGG | (unsigned long long)Q2);
        s_gbase = G2 ? atomicAdd(p.cand_cnt + i, G2) : 0u;   // cand_cnt was reset by pass 2: slot counter here
      }
      unsigned pe = 0;
      if (Q2 > 0 && t > ts) {                           // ties in this tile: how many ties precede it?
        int hi = t - 1;
        const uint64_t t_start = globaltimer_ns();
        while (hi >= ts && pe < need_eq) {              // once need_eq earlier ties exist, nothing here is selected
          const int s2 = hi - lane;
          unsigned long long d = SP_AGG;                // lanes below the tensor's first tile: neutral
          if (s2 >= ts) {
            do {
              d = ld_desc(p.desc + s2);
              if ((d >> 62) == 0ull && globaltimer_ns() - t_start > p.timeout_ns) {   // never hang the GPU
                atomicExch(p.status, EG_ERR_TIMEOUT);
                d = SP_AGG;
              }
            } while ((d >> 62) == 0ull);
          }
          unsigned ce = (s2 >= ts) ? (unsigned)(d & 0xFFFFFFFFull) : 0u;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) ce += __shfl_xor_sync(0xffffffffu, ce, o);
          pe += ce;
          hi -= 32;
        }
      }
      if (lane == 0) s_pe = pe;
    }
    __syncthreads();
    unsigned og = s_gbase, oe = s_pe;
    for (int w = 0; w < warp; ++w) {
      og += wg[w];
      oe += we[w];
    }
    og += gi - g;
    oe += qi - q;
    const size_t ro = (size_t)p.t_rec_off[i];
    bool touched = false;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      int pos = -1;
      if (fe & (1u << e)) {                             // ties: the need_eq lowest indices, slots [0, need_eq)
        if (oe < need_eq) pos = (int)oe;
        ++oe;
      } else if (fg & (1u << e)) {                      // every key > tau
        pos = (int)(need_eq + og++);
      }
      if (pos >= 0 && pos < k) {
        const float val = a.v[e];
        const float idxw = __int_as_float(first + tid * EG_VEC + e);
        p.rec_to_l[ro + pos] = val;
        p.rec_to_l[ro + k + pos] = idxw;
        if (p.rec_to_r != nullptr) {                    // null on a 2-rank ring: the one neighbour reads one copy
          p.rec_to_r[ro + pos] = val;
          p.rec_to_r[ro + k + pos] = idxw;
        }
        b.v[e] = val;                                   // prev[idx] <- value sent (spevent.cpp:407-413)
        touched = true;
      }
    }
    if (touched) st_f8(p.prev + base, b);
  }
  // ---- publish: per-tensor sequence numbers (+ step-done flag in iter-sync mode) -------------
  __syncthreads();
  if (tid == 0) {
    __threadfence_system();
    const unsigned prev = atomicAdd(p.ticket, 1u);
    s_last = (prev == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence_system();
  for (int i = tid; i < p.tab.n_tensors; i += EG_THREADS) {
    if (p.fire[i]) {
      st_release_sys(p.seq_to_l + i, (uint32_t)step);
      if (p.seq_to_r != nullptr) st_release_sys(p.seq_to_r + i, (uint32_t)step);
    }
  }
  __syncthreads();
  if (tid == 0) {
    *p.ticket = 0u;
    fence_sys();
    st_release_sys(p.done_to_l, (uint32_t)step);
    if (p.done_to_r != nullptr) st_release_sys(p.done_to_r, (uint32_t)step);
  }
}

// ---------------------------------------------------------------- stand-alone receive kernel
// (the product path runs sparse_apply_prologue inside the mix+SGD kernel; this launch exists for unit tests and for
// callers that keep the replicas up to date without stepping)
__global__ void __launch_bounds__(EG_THREADS, 4) sparse_apply_kernel(const SparseParams p) {
  sparse_apply_prologue(p, p.ticket + 2);
}

// ------------------------------------------------------------------------------------------
int sparse_select_grid(int n_tiles, int max_grid) {
  // blocked ranges of at most SP_MAX_OWN tiles per CTA for the two histogram passes
  int g = max_grid;
  const int need = (n_tiles + SP_MAX_OWN - 1) / SP_MAX_OWN;
  if (g < need) g = need;
  if (g > n_tiles) g = n_tiles;
  return g < 1 ? 1 : g;
}

cudaError_t launch_sparse_select_push(const SparseParams& p, int grid, cudaStream_t s) {
  eg_count_launch(EG_FAM_SPARSE, 3);
  const int hg = sparse_select_grid(p.tab.n_tiles, grid);
  sparse_hist_kernel<<<hg, EG_THREADS, 0, s>>>(p);
  sparse_cand_kernel<<<hg, EG_THREADS, 0, s>>>(p);
  sparse_compact_kernel<<<grid, EG_THREADS, 0, s>>>(p);      // persistent, co-resident: look-back needs progress
  return cudaGetLastError();
}

cudaError_t launch_sparse_apply(const SparseParams& p, int grid, cudaStream_t s) {
  eg_count_launch(EG_FAM_SPARSE, 1);
  sparse_apply_kernel<<<grid, EG_THREADS, 0, s>>>(p);
  return cudaGetLastError();
}

}  // namespace egb
