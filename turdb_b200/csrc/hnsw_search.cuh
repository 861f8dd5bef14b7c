// hnsw_search.cuh — the traversal kernel: greedy upper-level descent + level-0 beam search
// (PersistentHnswIndex::search, src/hnsw/mod.rs:1092-1174; greedy_search src/hnsw/search.rs:259-309;
// beam_search src/hnsw/search.rs:311-350).
//
// One CTA ("team" of W warps) owns one query at a time; CTAs are persistent and pull queries from an
// atomic counter.  Warp 0 (the leader) runs the reference's control flow on one sorted ef-slot list and stays
// out of the data path; warps 1..W-1 (helpers) gather and reduce.  Per hop the leader
//   (1) picks the closest unexpanded entry of the list (== candidates.pop() that passes d <= worst) and the
//       runner-up,
//   (2) if the runner-up of the PREVIOUS hop is this hop's node (81 % of hops), finds its unvisited neighbours
//       already filtered: while the helpers gathered the previous hop, the leader took the runner-up's adjacency
//       row and ran it through the exact visited set in shared memory as if it were this hop; on a miss the
//       speculative keys are taken back (visited_undo restores the table exactly) and the row is filtered now,
// then ALL warps of the team
//   (3) issue one TMA bulk copy per unvisited neighbour vector (cp.async.bulk -> shared memory staging,
//       mbarrier completion); vectors that do not fit the first round are prefetched into L2 meanwhile,
// the helpers
//   (4) reduce distances in the reference's AVX2 lane order (bit-identical values), chunks of 8 vectors each,
// and the leader
//   (5) merges the <=32 new (distance, id) pairs into the sorted list by rank counting, in place.
//
// Single-list equivalence with the reference's two heaps: SURVEY.md Appendix D / DESIGN.md §5.
#pragma once

#include "common.cuh"

// Measured and dropped: a double-buffered list merge (2 x 8 B x ef of shared memory) — the in-place merge in register
// batches below needs half the list memory (what lets 5 queries stay resident per SM at dim 384) and is also faster.

// Measured and dropped: per-thread 16 B cp.async (LDGSTS) gathers instead of one TMA bulk copy per vector — the LDGSTS
// issue stalls ~2.6k cycles per 8-vector chunk against ~0.9k for eight bulk copies, 25-33 % slower at 1M x 384 and
// 1M x 128 on B200.

// 1: vectors of a hop that do not fit the first gather round are prefetched into L2 during that round
#ifndef TURDB_R2_PREFETCH
#define TURDB_R2_PREFETCH 1
#endif

// Measured and dropped: splitting the bulk-copy issue of a second-round chunk between its owner and an idle
// helper (through a "slots free" mbarrier) — 3 % slower at 1M x 384 than the owner issuing alone.

// resident CTAs per SM the register allocation is bounded for (8 -> 64 registers per thread at 128 threads)
#ifndef TURDB_MIN_CTAS
#define TURDB_MIN_CTAS 5
#endif

// Measured and dropped: gathering FP32 rows four at a time with the TMA tensor copy's four-row gather mode (DESIGN.md §4.1)
// — parity-green but slower than the bulk copies (1M x 384: 9.94 vs 8.14 ms; 1M x 128: 5.18 vs 4.74 ms on B200): the issue
// phase does not shrink and the reduce over piece-split rows grows.

// Rows up to this many bytes are traversed by the direct form (one warp per query, hnsw_search_warp_kernel) unless the
// caller forces a form (turdb_cuda_index_set_traversal_form)
#ifndef TURDB_DIRECT_MAX_ROW_BYTES
#define TURDB_DIRECT_MAX_ROW_BYTES 1024
#endif
#ifndef TURDB_DIRECT_MAX_ROWS_PER_HOP
#define TURDB_DIRECT_MAX_ROWS_PER_HOP 10.0
#endif

namespace turdb {

constexpr uint32_t kDone = 0xFFFFFFFFu;
constexpr uint32_t kInsLevels = 16;   // levels 0..15 (select_level caps at 15, operations.rs:76-79)
constexpr uint32_t kInsSelMax = 64;   // m0 = 2 M <= 64
#ifndef TURDB_MERGE_BATCH
#define TURDB_MERGE_BATCH 4
#endif
constexpr int kMergeBatch = TURDB_MERGE_BATCH;

// fixed offsets of the small per-query arrays (the variable-size ones follow: list, filtered window, query, table, staging)
constexpr uint32_t kOffBar = 0, kOffCtl = 32, kOffCand = 64, kOffList = 576;

struct TeamLayout {
  uint32_t off_q, off_clist, off_hash, off_stage;
  uint32_t team_bytes;
  uint32_t n_groups;   // staging groups of 8 slots (1..4), one mbarrier each
  uint32_t stride;     // bytes between staging slots; stride/4 == 8 (mod 32) -> conflict-free quads
  uint32_t vec_bytes;  // ds * 4
  // a vector streams through its slot in n_segs pieces of seg_steps AVX steps (32 B each); the last piece
  // also carries the < 8-element tail.  The quad's accumulators live in registers across pieces.
  uint32_t n_segs, seg_steps;
  uint32_t hash_bits;  // shared visited table has 1 << hash_bits slots
  // compact table (hash16 != 0): 16-bit entries = (displacement+1) << rem_bits | remainder of a
  // bijective hash of the id, so an entry still identifies exactly one node (exact set, half the bytes)
  uint32_t hash16;
  uint32_t rem_bits;   // key_bits - hash_bits
  uint32_t key_bits;   // ceil(log2(n)), >= hash_bits
};

// Feedback from past launches, one record per ceil(log2(ef)) class: the largest visited set any query produced (sizes
// the shared-memory table) and the level-0 totals whose ratio is the new rows gathered per expansion (picks the form).
struct TraversalStats {
  uint32_t vis_max, pad;
  unsigned long long sum_dist, sum_exp;
};

struct SearchArgs {
  DeviceIndex ix;
  TeamLayout lay;
  const float* queries;  // [nq][dim]
  uint32_t nq, k, ef;
  uint64_t* out_row_ids;  // [nq][k]
  uint32_t* out_node_ids; // [nq][k] or null
  float* out_dist;        // [nq][k]
  uint32_t* out_counts;   // [nq]
  uint32_t* out_stats;    // [nq][4] or null
  uint32_t* work_counter; // zeroed before launch
  uint32_t* overflow_count;  // queries whose shared visited table could not place a key
  uint32_t* overflow_list;   // [nq]
  uint32_t* global_visited;  // fallback pass: [CTAs][vis_words] bitsets
  uint32_t vis_words;
  unsigned long long* dbg;   // optional [16] cycle counters (diagnostics), null in production
  // rows the traversal gathers: the FP32 arena (row_bytes == ds * 4) or, for the SQ8 kernels, the code arena
  const uint8_t* rows;
  uint32_t row_bytes;        // bytes between rows == bytes copied per row (multiple of 16)
  // search_filtered (search.rs:352-398): one bit per node; candidates that do not fit the shared window
  const uint64_t* visible;   // null => unfiltered search
  uint2* f_ovf;              // [CTAs][f_ocap] (distance bits, id) overflow of the candidate window
  uint32_t f_ocap;
  TraversalStats* tstats;    // optional: what this ef class's queries looked like (sizes and shapes the next launch)
  // INSERT kernels (graph_insert.inl): query q is node ins_first + q; per level l <= ins_levels[q] the beam's nearest
  // ins_m0 (l == 0) / ins_m ids go to ins_sel[q][l][0..ins_cnt[q][l])
  uint32_t ins_first, ins_m, ins_m0;
  const uint8_t* ins_levels;  // [nq]
  uint32_t* ins_sel;          // [nq][kInsLevels][kInsSelMax]
  uint8_t* ins_cnt;           // [nq][kInsLevels]
};

// Per-team shared state handed to every warp.
struct Team {
  // chunk c of a request is gathered and reduced by owner(c): with helpers, warp 0 (the leader) keeps out of
  // the data path and spends the gather time preparing the next hop (speculative visited filtering)
  // A request has at most 4 chunks (32 candidates); their staging group (c % n_groups) and whether this warp
  // owns them are tabulated once per kernel (grp_pack: 2 bits per chunk, own_mask: 1 bit per chunk) so that
  // the per-hop loops hold no integer division.
  __device__ __forceinline__ bool owns(uint32_t c) const { return (own_mask >> c) & 1u; }
  __device__ __forceinline__ uint32_t group_of(uint32_t c) const { return (grp_pack >> (2 * c)) & 3u; }
  __device__ __forceinline__ void tabulate() {
    grp_pack = 0;
    own_mask = 0;
    for (uint32_t c = 0; c < 4; ++c) {
      const uint32_t g = c % n_groups;
      const uint32_t o = n_warps == 1 ? 0u : 1u + g % (n_warps - 1);
      grp_pack |= g << (2 * c);
      own_mask |= (o == warp ? 1u : 0u) << c;
    }
  }
  uint32_t grp_pack, own_mask;
  uint32_t lane, warp, n_warps;
  uint32_t bar0;             // shared address of mbarrier 0 (8 B apart)
  volatile uint32_t* ctl;    // [0] = m of the current request or kDone, [1] = work item
  const float* q;            // staged query
  uint32_t* cand_ids;        // [32] ids whose distances are requested
  float* cand_d;             // [32] results
  const uint8_t* stage;
  uint32_t stage_u32;
  uint32_t stride, vec_bytes, n_groups, n_segs, seg_steps;
  const uint8_t* rows;       // gather source, vec_bytes apart
  uint32_t phases;           // per-warp parity bits of the groups this warp owns
  float qnorm;
  uint32_t c_issue, c_wait, c_comp;  // diagnostics: cycles spent by this warp per phase
  bool dbg;
};

// Every warp of the team calls this between the two team barriers of a request: chunk c (candidates
// 8c..8c+7) uses staging group c % G and is handled by that group's owner (Team::owns).  A chunk's vectors stream through
// their slots in n_segs pieces; a warp keeps one piece of every group it owns in flight, reduces a piece as
// soon as it lands and immediately requests the next one (of the same chunk, or the first piece of the next
// chunk mapped to that group).
template <int METRIC>
__device__ __forceinline__ void team_distances_pieces(const DeviceIndex& ix, Team& t, uint32_t m) {
  const uint32_t lane = t.lane, p = lane & 3, G = t.n_groups, S = t.n_segs;
  const uint32_t nchunks = (m + 7) >> 3;
  const uint32_t steps = ix.dim >> 3;
  auto seg_lo = [&](uint32_t sgm) { return min(steps, sgm * t.seg_steps); };
  auto issue = [&](uint32_t c, uint32_t sgm) {
    const uint32_t g = t.group_of(c);
    const uint32_t bar = t.bar0 + 8 * g;
    const uint32_t cnt = min(8u, m - 8 * c);
    const uint32_t b0 = seg_lo(sgm) * 32;
    const uint32_t b1 = (sgm + 1 == S) ? t.vec_bytes : seg_lo(sgm + 1) * 32;
    if (lane == 0) mbar_expect_tx(bar, cnt * (b1 - b0));
    __syncwarp();
    if (lane < cnt && b1 > b0) {
      const uint32_t id = t.cand_ids[8 * c + lane];
      bulk_g2s(t.stage_u32 + (g * 8 + lane) * t.stride, reinterpret_cast<const uint8_t*>(ix.arena + (size_t)id * ix.ds) + b0,
               b1 - b0, bar);
    }
  };
  long long t0 = t.dbg ? clock64() : 0;
  for (uint32_t c = 0; c < min(G, nchunks); ++c)
    if (t.owns(c)) issue(c, 0);
  if (t.dbg) t.c_issue += (uint32_t)(clock64() - t0);
  for (uint32_t c = 0; c < nchunks; ++c) {
    const uint32_t g = t.group_of(c);
    if (!t.owns(c)) continue;
    const uint32_t slot = 8 * c + (lane >> 2);
    float nb = 0.f;
    if (METRIC == kCosine && slot < m) nb = __ldg(ix.norm2 + t.cand_ids[slot]);
    const uint8_t* sb = t.stage + (g * 8 + (lane >> 2)) * t.stride;
    uint64_t acc = 0ull;
    float raw = 0.f, first = 0.f;
    for (uint32_t sgm = 0; sgm < S; ++sgm) {
      long long w0 = t.dbg ? clock64() : 0;
      mbar_wait(t.bar0 + 8 * g, (t.phases >> g) & 1u);
      long long w1 = t.dbg ? clock64() : 0;
      t.c_wait += (uint32_t)(w1 - w0);
      t.phases ^= (1u << g);
      const uint32_t s0 = seg_lo(sgm), s1 = (sgm + 1 == S) ? steps : seg_lo(sgm + 1);
      if (sgm == 0) first = *reinterpret_cast<const float*>(sb);
      const uint64_t* av = reinterpret_cast<const uint64_t*>(t.q + 8 * s0) + p;
      const uint64_t* bv = reinterpret_cast<const uint64_t*>(sb) + p;
      acc = (METRIC == kL2) ? quad_accum<true>(acc, av, bv, s1 - s0) : quad_accum<false>(acc, av, bv, s1 - s0);
      if (sgm + 1 == S) {
        const float* bt = reinterpret_cast<const float*>(sb) + 8 * (s1 - s0);
        raw = (METRIC == kL2) ? quad_finish<true>(acc, t.q + 8 * steps, bt, ix.dim & 7)
                              : quad_finish<false>(acc, t.q + 8 * steps, bt, ix.dim & 7);
      }
      __syncwarp();
      if (t.dbg) t.c_comp += (uint32_t)(clock64() - w1);
      if (sgm + 1 < S) issue(c, sgm + 1);
      else if (c + G < nchunks) issue(c + G, 0);
    }
    if (p == 0 && slot < m) {
      float d = raw;
      if (METRIC == kIP) d = -raw;  // inner_product_avx2, distance.rs:240-242
      if (METRIC == kCosine) d = cosine_finish(raw, t.qnorm, nb);
      if (first == INFINITY) d = INFINITY;  // absent vector (+inf row): get_vector -> None, mod.rs:1111-1121
      t.cand_d[slot] = d;
    }
  }
}

// Whole-vector form (n_segs == 1): same dealing of chunks to groups and warps, one bulk copy per vector.
template <int METRIC, bool SQ8>
__device__ __forceinline__ void team_distances_whole(const DeviceIndex& ix, Team& t, uint32_t m) {
  const uint32_t lane = t.lane, p = lane & 3, G = t.n_groups;
  const uint32_t nchunks = (m + 7) >> 3;
  auto issue = [&](uint32_t c) {
    const uint32_t g = t.group_of(c);
    const uint32_t bar = t.bar0 + 8 * g;
    const uint32_t cnt = min(8u, m - 8 * c);
    if (lane == 0) mbar_expect_tx(bar, cnt * t.vec_bytes);
    __syncwarp();
    if (lane < cnt) {
      const uint32_t id = t.cand_ids[8 * c + lane];
      bulk_g2s(t.stage_u32 + (g * 8 + lane) * t.stride, t.rows + (size_t)id * t.vec_bytes, t.vec_bytes, bar);
    }
  };
  long long t0 = t.dbg ? clock64() : 0;
  // Round 1 (the first min(m, 8G) vectors): a bulk copy is issued lane by lane (ELECT / R2UR / UBLKCP, ~100
  // cycles each), so the copies are dealt to ALL warps of the team, the leader included (vector v to warp
  // v % W, one lane each), which divides that latency by W.  The owner of a chunk arms the chunk's barrier
  // with the byte count; completions that land before the arming only run the transaction count negative.
  {
    const uint32_t m1 = min(m, 8 * G);
    for (uint32_t c = 0; c < min(G, nchunks); ++c)
      if (t.owns(c) && lane == 0) mbar_expect_tx(t.bar0 + 8 * c, min(8u, m - 8 * c) * t.vec_bytes);
    const uint32_t v = t.warp + t.n_warps * lane;
    if (v < m1) {
      const uint32_t id = t.cand_ids[v];  // chunk v >> 3 < G uses group v >> 3, slot v & 7: staging slot v
      bulk_g2s(t.stage_u32 + v * t.stride, t.rows + (size_t)id * t.vec_bytes, t.vec_bytes, t.bar0 + 8 * (v >> 3));
    }
#if TURDB_R2_PREFETCH
    // The vectors that have to wait for a second round (no free staging slot yet) are pulled into L2 now, by
    // the leader (it has slack): their bulk copies will then pay an L2 hit instead of a second DRAM round
    // trip.  Same DRAM bytes — every one of them is read exactly once, for certain, a little later.
    if (t.warp == 0 && t.n_warps >= 3 && m1 + lane < m)  // a 2-warp team has no slack on the leader (measured)
      bulk_prefetch_l2(t.rows + (size_t)t.cand_ids[m1 + lane] * t.vec_bytes, t.vec_bytes);
#endif
  }
  if (t.dbg) t.c_issue += (uint32_t)(clock64() - t0);
  for (uint32_t c = 0; c < nchunks; ++c) {
    const uint32_t g = t.group_of(c);
    if (!t.owns(c)) continue;
    const uint32_t slot = 8 * c + (lane >> 2);
    float nb = 0.f;
    if (METRIC == kCosine && slot < m) nb = __ldg(ix.norm2 + t.cand_ids[slot]);
    long long w0 = t.dbg ? clock64() : 0;
    mbar_wait(t.bar0 + 8 * g, (t.phases >> g) & 1u);
    long long w1 = t.dbg ? clock64() : 0;
    t.c_wait += (uint32_t)(w1 - w0);
    t.phases ^= (1u << g);
    const uint8_t* bs = t.stage + (g * 8 + (lane >> 2)) * t.stride;
    const float* b = reinterpret_cast<const float*>(bs);
    float raw;
    if (SQ8) raw = (METRIC == kL2) ? quad_sq8<0>(t.q, bs, ix.dim, p) : quad_sq8<1>(t.q, bs, ix.dim, p);
    else raw = (METRIC == kL2) ? quad_l2sq(t.q, b, ix.dim, p) : quad_dot(t.q, b, ix.dim, p);
    if (p == 0 && slot < m) {
      float d = raw;
      if (METRIC == kIP) d = -raw;  // inner_product_avx2, distance.rs:240-242
      if (METRIC == kCosine) d = cosine_finish(raw, t.qnorm, nb);
      // absent vector (uploaded as a +inf row; SQ8: min == +inf): get_vector -> None => INFINITY, mod.rs:1111-1121
      if ((SQ8 ? *reinterpret_cast<const float*>(bs + ((ix.dim + 3) & ~3u)) : b[0]) == INFINITY) d = INFINITY;
      t.cand_d[slot] = d;
    }
    __syncwarp();
    if (t.dbg) t.c_comp += (uint32_t)(clock64() - w1);
    if (c + G < nchunks) issue(c + G);
  }
}

template <int METRIC, bool SQ8>
__device__ __forceinline__ void team_distances(const DeviceIndex& ix, Team& t, uint32_t m) {
  if (SQ8) {  // code rows are short: always the whole-row form (the host never splits them)
    team_distances_whole<METRIC, true>(ix, t, m);
    return;
  }
  if (t.n_segs == 1) team_distances_whole<METRIC, false>(ix, t, m);
  else team_distances_pieces<METRIC>(ix, t, m);
}

// Leader side of a request: publish m, run the team's distance pass, return this lane's distance.
// `overlap` runs on the leader between the two barriers, i.e. while the helper warps gather and reduce.
template <int METRIC, bool SQ8, typename F>
__device__ __forceinline__ float leader_request(const DeviceIndex& ix, Team& t, uint32_t m, F&& overlap) {
  if (t.lane == 0) t.ctl[0] = m;
  __syncthreads();
  team_distances<METRIC, SQ8>(ix, t, m);  // the leader only takes its share of the first round's copies
  overlap();
  __syncthreads();
  return t.lane < m ? t.cand_d[t.lane] : INFINITY;
}
template <int METRIC, bool SQ8>
__device__ __forceinline__ float leader_request(const DeviceIndex& ix, Team& t, uint32_t m) {
  return leader_request<METRIC, SQ8>(ix, t, m, [] {});
}

// ---- direct mode: ONE WARP per query, neighbour rows gathered straight into registers --------------------
// For short rows (dim <= ~256) a hop moves only a few KB, and what bounds the kernel is how many hops an SM
// keeps in flight, not how fast one hop runs.  The direct form drops the team: no staging slots, no mbarriers,
// no CTA barriers — a 32-thread CTA per query (16-20 resident per SM), the registers are the landing zone.
// A quad of lanes owns one neighbour row per pass (8 rows per pass); lane p of the quad loads the 8 bytes
// (elements 8t+2p, 8t+2p+1) of AVX step t with one LDG.64, so the quad reads one 32 B sector per step and every
// lane's accumulator is exactly the reference's AVX2 lane pair (distance.rs:105-129).  A row streams through in
// units of 8 steps (64 floats, 8 register pairs per lane); one unit is in flight per warp, and the rest of the request
// is prefetched into L2 (TURDB_DIRECT_PREFETCH).
// step S of a unit: base + 32 S bytes, the offset folded into the instruction (a register operand per load would
// cost an address register pair each)
template <int S, int US>
struct LoadSteps {
  static __device__ __forceinline__ void run(uint64_t (&b)[US], const uint64_t* base, uint32_t ns) {
    if ((uint32_t)S < ns) asm volatile("ld.global.nc.L1::no_allocate.b64 %0, [%1+%2];" : "=l"(b[S]) : "l"(base), "n"(32 * S));
    LoadSteps<S + 1, US>::run(b, base, ns);
  }
};
template <int US>
struct LoadSteps<US, US> {
  static __device__ __forceinline__ void run(uint64_t (&)[US], const uint64_t*, uint32_t) {}
};

// Measured and dropped: prefetching the rows of the speculated next hop into L2 during the current hop — no gain in the
// direct form (2.648 vs 2.647 ms), 5 % slower in the staged form (3.16 vs 3.00 ms) at 2M x 128 clustered / 1M x 128
// SIFT-like on B200: the 128-d kernel waits on dependent instructions, not on the rows.
// Measured and dropped: direct-form landing zones of 16 steps x 1, 8 x 2, 8 x 3 and 4 x 2 units in flight — all slower
// or spilling against 8 x 1.
#ifndef TURDB_DIRECT_DBG
#define TURDB_DIRECT_DBG 0
#endif
// 1: rows of a request beyond the first pass (candidates 8..m-1) are prefetched into L2 when the request starts,
// one 128 B line per lane and instruction: their loads then pay an L2 hit instead of a second and third DRAM
// round trip, without holding registers for them meanwhile.  Same DRAM bytes: every line is consumed for certain.
#ifndef TURDB_DIRECT_PREFETCH
#define TURDB_DIRECT_PREFETCH 1
#endif

template <int METRIC, typename F>
__device__ __forceinline__ float warp_request(const DeviceIndex& ix, Team& t, uint32_t m, F&& overlap) {
  constexpr int US = 8;  // steps (of 8 floats) per unit: the landing zone is 2 * US registers
  const uint32_t lane = t.lane, p = lane & 3, qd = lane >> 2;
  const uint32_t steps = ix.dim >> 3, ntail = ix.dim & 7;
  const uint32_t nch = max(1u, (steps + US - 1) / US);
  const bool full = steps != 0 && steps % US == 0;  // every unit carries US steps: the loops below run unpredicated
  const uint32_t npass = (m + 7) >> 3, nunits = npass * nch;
  uint64_t b[US];
  __syncwarp();  // cand_ids[0..m) were written by lanes 0..m-1; every quad reads them (the staged form has a CTA barrier here)
  // Quads beyond the request's last candidate gather (and reduce) that last candidate again: every lane then runs
  // the same unpredicated instruction stream; their result is discarded.
  uint32_t l_pass = 0, l_ch = 0;  // next unit to load
  auto load = [&] {
    const uint32_t id = t.cand_ids[min(8 * l_pass + qd, m - 1)];
    const uint64_t* src = reinterpret_cast<const uint64_t*>(t.rows + (size_t)id * t.vec_bytes) + 4 * US * l_ch + p;
    if (full) LoadSteps<0, US>::run(b, src, US);
    else LoadSteps<0, US>::run(b, src, min((uint32_t)US, steps - US * l_ch));
    if (++l_ch == nch) {
      l_ch = 0;
      ++l_pass;
    }
  };
  uint32_t c_pass = 0, c_ch = 0;  // next unit to reduce
  uint64_t acc = 0ull;
  float out = INFINITY, first = 0.f;
  auto consume = [&] {
    const uint64_t* av = reinterpret_cast<const uint64_t*>(t.q + 8 * US * c_ch) + p;
    if (full) {
      if (c_ch == 0) first = __uint_as_float((uint32_t)b[0]);  // element 0 of the row, in the quad's lane 0
#pragma unroll
      for (int s = 0; s < US; ++s) {
        if (METRIC == kL2) {
          const uint64_t d = sub2(av[4 * s], b[s]);
          acc = fma2(d, d, acc);
        } else {
          acc = fma2(av[4 * s], b[s], acc);
        }
      }
    } else {
      const uint32_t ns = min((uint32_t)US, steps - US * c_ch);
      if (c_ch == 0) first = ns ? __uint_as_float((uint32_t)b[0]) : 0.f;
#pragma unroll
      for (int s = 0; s < US; ++s)
        if ((uint32_t)s < ns) {
          if (METRIC == kL2) {
            const uint64_t d = sub2(av[4 * s], b[s]);
            acc = fma2(d, d, acc);
          } else {
            acc = fma2(av[4 * s], b[s], acc);
          }
        }
    }
    if (++c_ch == nch) {
      // row complete: horizontal sum in the reference's order, the unfused scalar tail, the metric's epilogue
      float r = quad_hsum(unpack2(acc));
      const uint32_t id = t.cand_ids[min(8 * c_pass + qd, m - 1)];
      if (ntail | (steps == 0)) {
        const float* row = reinterpret_cast<const float*>(t.rows + (size_t)id * t.vec_bytes);
        for (uint32_t i = 0; i < ntail; ++i) {
          const float a = t.q[8 * steps + i], bv = __ldg(row + 8 * steps + i);
          if (METRIC == kL2) {
            const float d = __fsub_rn(a, bv);
            r = __fadd_rn(r, __fmul_rn(d, d));
          } else {
            r = __fadd_rn(r, __fmul_rn(a, bv));
          }
        }
        if (steps == 0) first = __ldg(row);
      }
      float d = r;
      if (METRIC == kIP) d = -r;  // inner_product_avx2, distance.rs:240-242
      if (METRIC == kCosine) d = cosine_finish(r, t.qnorm, __ldg(ix.norm2 + id));
      // absent vector (uploaded as a +inf row): get_vector -> None => distance INFINITY for every metric, mod.rs:1111-1121
      if (__shfl_sync(kFullMask, first, lane & ~3u) == INFINITY) d = INFINITY;
      // lane i of the warp receives candidate i: candidate 8*pass + j lives in quad j
      const float v = __shfl_sync(kFullMask, d, (lane & 7) << 2);
      if ((lane >> 3) == c_pass) out = v;
      acc = 0ull;
      c_ch = 0;
      ++c_pass;
    }
  };
  if (nunits != 0) load();
#if TURDB_DIRECT_PREFETCH
  if (nunits > 1) {
    // everything the first unit does not cover is pulled into L2 now, one 128 B line per lane and instruction
    // (whole rows of the later candidates; with rows longer than one unit, the rest of every row)
    const uint32_t r0 = nch == 1 ? 8u : 0u;
    const uint32_t lpr = ((t.vec_bytes + 127) >> 7) + ((t.vec_bytes & 127) ? 1u : 0u);  // lines a row can touch
    const uint32_t sh = 32 - __clz(lpr - 1), total = (m - min(m, r0)) << sh;             // rounded up to a power of two
    for (uint32_t j = lane; j < total; j += 32) {
      const uint32_t r = r0 + (j >> sh), l = j & ((1u << sh) - 1);
      const uint8_t* row = t.rows + (size_t)t.cand_ids[r] * t.vec_bytes;
      const uintptr_t a = (reinterpret_cast<uintptr_t>(row) & ~(uintptr_t)127) + 128 * l;
      if (a < reinterpret_cast<uintptr_t>(row) + t.vec_bytes) asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
    }
  }
#endif
  overlap();
  for (uint32_t u = 0; u < nunits; ++u) {
    consume();
    if (u + 1 < nunits) load();
  }
  __syncwarp();  // all reads of cand_ids are done before the caller reuses it
  return lane < m ? out : INFINITY;
}

// One request, either form.
template <int METRIC, bool SQ8, bool DIRECT, typename F>
__device__ __forceinline__ float request(const DeviceIndex& ix, Team& t, uint32_t m, F&& overlap) {
  if (DIRECT) return warp_request<METRIC>(ix, t, m, overlap);
  return leader_request<METRIC, SQ8>(ix, t, m, overlap);
}
template <int METRIC, bool SQ8, bool DIRECT>
__device__ __forceinline__ float request(const DeviceIndex& ix, Team& t, uint32_t m) {
  return request<METRIC, SQ8, DIRECT>(ix, t, m, [] {});
}
template <bool DIRECT>
__device__ __forceinline__ void team_sync() {
  if (DIRECT) __syncwarp();
  else __syncthreads();
}

// Exact visited set, called by all 32 lanes of the leader with one (distinct) id per active lane.
// Returns 1 = newly inserted, 0 = already present (or inactive lane), 2 = table cannot place the key
// (the query is then redone by the global-bitset pass).
//   GLOBAL : one bit per node in global memory (atomicOr).
//   shared : open addressing, linear probing, no atomics: only this warp touches the table, so a round is
//            "read slot; if empty write my entry; re-read: did my write survive?".  All reads of a round
//            precede its writes (same instruction), and rows never repeat an id (deduplicated at upload), so
//            two lanes can only collide with DIFFERENT entries and the loser simply probes on.
//     32-bit entries hold the id.  16-bit entries: h = id * odd (mod 2^key_bits) is a bijection; home = top
//     hash_bits of h; the entry stores the low rem_bits of h plus (displacement + 1), which together name h
//     and therefore the id — an exact set in half the bytes.
// *where (optional) receives the table position a newly inserted key went to, for visited_undo.
template <bool GLOBAL>
__device__ __forceinline__ uint32_t visited_insert(uint32_t* tab, uint32_t id, bool active, const TeamLayout& L,
                                                   uint32_t* where = nullptr) {
  if (GLOBAL) {
    if (!active) return 0u;
    const uint32_t bit = 1u << (id & 31);
    if (where) *where = id;
    return (atomicOr(tab + (id >> 5), bit) & bit) == 0 ? 1u : 0u;
  }
  const uint32_t mask = (1u << L.hash_bits) - 1;
  constexpr uint32_t kPending = 3u;
  uint32_t res = active ? kPending : 0u;
  if (L.hash16) {
    volatile unsigned short* t16 = reinterpret_cast<volatile unsigned short*>(tab);
    const uint32_t h = (id * 0x9E3779B1u) & ((1u << L.key_bits) - 1);
    const uint32_t home = h >> L.rem_bits, rem = h & ((1u << L.rem_bits) - 1);
    const uint32_t max_disp = (1u << (16 - L.rem_bits)) - 1;  // displacement+1 must fit
    uint32_t disp = 0;
    while (__any_sync(kFullMask, res == kPending)) {
      bool wrote = false;
      uint32_t slot = 0;
      unsigned short want = 0;
      if (res == kPending) {
        if (disp >= max_disp) {
          res = 2u;
        } else {
          slot = (home + disp) & mask;
          want = (unsigned short)(((disp + 1) << L.rem_bits) | rem);
          const unsigned short e = t16[slot];
          if (e == want) res = 0u;
          else if (e == 0) {
            t16[slot] = want;
            wrote = true;
          } else {
            ++disp;
          }
        }
      }
      __syncwarp();
      if (wrote) {
        if (t16[slot] == want) {
          res = 1u;
          if (where) *where = slot;
        } else {
          ++disp;
        }
      }
      __syncwarp();
    }
    return res;
  }
  volatile uint32_t* t32 = tab;
  uint32_t slot = (id * 0x9E3779B1u) >> (32 - L.hash_bits);
  while (__any_sync(kFullMask, res == kPending)) {
    bool wrote = false;
    if (res == kPending) {
      const uint32_t e = t32[slot];
      if (e == id) res = 0u;
      else if (e == kInvalid) {
        t32[slot] = id;
        wrote = true;
      } else {
        slot = (slot + 1) & mask;
      }
    }
    __syncwarp();
    if (wrote) {
      if (t32[slot] == id) {
        res = 1u;
        if (where) *where = slot;
      } else {
        slot = (slot + 1) & mask;
      }
    }
    __syncwarp();
  }
  return res;
}

// Takes back the keys one visited_insert call inserted (`inserted` = that call returned 1 for this lane,
// `where` = its position).  Exact as long as nothing was inserted since: keys only ever go to EMPTY slots, so
// emptying the newest ones cannot cut the probe sequence of any older key.
template <bool GLOBAL>
__device__ __forceinline__ void visited_undo(uint32_t* tab, bool inserted, uint32_t where, const TeamLayout& L) {
  if (inserted) {
    if (GLOBAL) atomicAnd(tab + (where >> 5), ~(1u << (where & 31)));
    else if (L.hash16) reinterpret_cast<volatile unsigned short*>(tab)[where] = 0;
    else reinterpret_cast<volatile uint32_t*>(tab)[where] = kInvalid;
  }
  __syncwarp();
}

// Merge up to 32 new (d, id) pairs (one per `elig` lane) into the ascending list src[head, len) -> dst[0, ..),
// keeping at most `cap` entries.  Old entries win distance ties; new ones tie-break by lane (stored order).
// EVICT: entries pushed past `cap` are appended to the global overflow `ovf` (they stay candidates) unless
// `drop_above` says they can never be expanded (d > drop_above); *o_min tracks the smallest overflowed distance.
// Returns the new length; *min_new = smallest position taken by a new entry (0xFFFFFFFF if none).
template <bool EVICT>
__device__ __forceinline__ uint32_t rank_merge(const float* src_d, const uint32_t* src_id, uint32_t head, uint32_t len,
                                               float* dst_d, uint32_t* dst_id, uint32_t cap, bool elig, float d,
                                               uint32_t id, uint32_t* tmp_ub, uint32_t lane, uint32_t* min_new,
                                               uint2* ovf, uint32_t* o_cnt, uint32_t o_cap, float* o_min,
                                               float drop_above, bool* o_overflow) {
  const uint32_t n_old = len - head;
  const uint32_t emask = __ballot_sync(kFullMask, elig);
  const uint32_t mp = __popc(emask);
  uint32_t ub = 0;
  if (elig) {
    uint32_t lo = 0, hi = n_old;
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (src_d[head + mid] <= d) lo = mid + 1;
      else hi = mid;
    }
    ub = lo;
    tmp_ub[__popc(emask & ((1u << lane) - 1))] = ub;
  }
  uint32_t rank = 0;
  for (uint32_t e = emask; e; e &= e - 1) {
    const uint32_t bsrc = __ffs(e) - 1;
    const float db = __shfl_sync(kFullMask, d, bsrc);
    rank += (db < d || (db == d && bsrc < lane)) ? 1u : 0u;
  }
  __syncwarp();
  const uint32_t o_base = EVICT ? *o_cnt : 0u;
  uint32_t kept_evicted = 0;
  float ev_min = INFINITY;
  auto place = [&](uint32_t np, float pd, uint32_t pid) {
    if (np < cap) {
      dst_d[np] = pd;
      dst_id[np] = pid;
    } else if (EVICT && !(pd > drop_above)) {
      const uint32_t o = o_base + (np - cap);
      if (o < o_cap) ovf[o] = make_uint2(__float_as_uint(pd), pid);
      else *o_overflow = true;
      kept_evicted += 1;
      ev_min = fminf(ev_min, pd);
    }
  };
  for (uint32_t i = lane; i < n_old; i += 32) {
    uint32_t sft = 0;
    for (uint32_t j = 0; j < mp; ++j) sft += (tmp_ub[j] <= i) ? 1u : 0u;
    place(i + sft, src_d[head + i], src_id[head + i]);
  }
  uint32_t my_np = 0xFFFFFFFFu;
  if (elig) {
    my_np = ub + rank;
    place(my_np, d, id);
    if (my_np >= cap) my_np = 0xFFFFFFFFu;
  }
  *min_new = __reduce_min_sync(kFullMask, my_np);
  if (EVICT) {
    // evicted entries are the largest of the merged sequence and the dropped ones its tail, so the kept
    // ones occupy consecutive overflow slots
    *o_cnt = o_base + __reduce_add_sync(kFullMask, kept_evicted);
#pragma unroll
    for (uint32_t off = 16; off >= 1; off >>= 1) ev_min = fminf(ev_min, __shfl_xor_sync(kFullMask, ev_min, off));
    *o_min = fminf(*o_min, ev_min);
    if (__any_sync(kFullMask, *o_overflow)) *o_overflow = true;
  }
  __syncwarp();
  return min(n_old + mp, cap);
}

template <int METRIC, bool GLOBAL_VISITED, bool FILTERED, bool SQ8, bool DIRECT, bool INSERT = false>
__device__ __forceinline__ void hnsw_search_body(const SearchArgs& a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const DeviceIndex& ix = a.ix;
  const uint32_t tid = threadIdx.x, nthreads = blockDim.x;
  const uint32_t lane = tid & 31, warp = tid >> 5;
  float* qs = reinterpret_cast<float*>(smem + a.lay.off_q);
  float* A_d = reinterpret_cast<float*>(smem + kOffList);  // result list (sorted, ef slots)
  uint32_t* A_id = reinterpret_cast<uint32_t*>(A_d + a.ef);
  float* B_d = reinterpret_cast<float*>(A_id + a.ef);             // second buffer: filtered search only
  uint32_t* B_id = reinterpret_cast<uint32_t*>(B_d + a.ef);
  float* C_d = reinterpret_cast<float*>(smem + a.lay.off_clist);  // filtered search: candidate window (x2)
  uint32_t* C_id = reinterpret_cast<uint32_t*>(C_d + a.ef);
  float* D_d = reinterpret_cast<float*>(C_id + a.ef);
  uint32_t* D_id = reinterpret_cast<uint32_t*>(D_d + a.ef);
  uint32_t* cand_ids = reinterpret_cast<uint32_t*>(smem + kOffCand);
  float* cand_d = reinterpret_cast<float*>(cand_ids + 32);
  uint32_t* tmp_ub = cand_ids + 64;
  uint32_t* cand_next = cand_ids + 96;  // ids of the speculatively prepared next request
  uint32_t* vis = GLOBAL_VISITED ? a.global_visited + (size_t)blockIdx.x * a.vis_words
                                 : reinterpret_cast<uint32_t*>(smem + a.lay.off_hash);
  const uint32_t hash_slots = 1u << a.lay.hash_bits;
  const uint32_t hash_limit = hash_slots - (hash_slots >> 3);  // 7/8 full -> overflow path

  Team t;
  t.lane = lane;
  t.warp = warp;
  t.n_warps = nthreads >> 5;
  t.bar0 = smem_u32(smem + kOffBar);
  t.ctl = reinterpret_cast<volatile uint32_t*>(smem + kOffCtl);
  t.q = qs;
  t.cand_ids = cand_ids;
  t.cand_d = cand_d;
  t.stage = smem + a.lay.off_stage;
  t.stage_u32 = smem_u32(t.stage);
  t.stride = a.lay.stride;
  t.vec_bytes = a.lay.vec_bytes;
  t.rows = a.rows;
  t.n_groups = a.lay.n_groups;
  t.n_segs = a.lay.n_segs;
  t.seg_steps = a.lay.seg_steps;
  t.phases = 0;
  t.qnorm = 0.f;
  t.c_issue = t.c_wait = t.c_comp = 0;
  t.dbg = (DIRECT && !TURDB_DIRECT_DBG) ? false : a.dbg != nullptr;  // the direct form's register budget has no room for the counters
  if (!DIRECT) t.tabulate();

  if (!DIRECT && tid == 0) {
    for (uint32_t g = 0; g < a.lay.n_groups; ++g) mbar_init(t.bar0 + 8 * g, 1);
    mbar_fence_init();
  }
  team_sync<DIRECT>();

  const uint32_t ef = a.ef;
  const uint32_t n_work = GLOBAL_VISITED ? *a.overflow_count : a.nq;

  for (;;) {
    if (tid == 0) t.ctl[1] = atomicAdd(a.work_counter, 1u);
    team_sync<DIRECT>();
    const uint32_t wi = t.ctl[1];
    if (wi >= n_work) break;
    const uint32_t qi = GLOBAL_VISITED ? a.overflow_list[wi] : wi;

    // ---- stage the query, clear the visited set (whole team) ----
    // INSERT: the "query" is the new node's own vector (insert_with_callback, mod.rs:999-1084), already in the arena
    const float* qg = INSERT ? ix.arena + (size_t)(a.ins_first + qi) * ix.ds : a.queries + (size_t)qi * ix.dim;
    const uint32_t target = INSERT ? a.ins_levels[qi] : 0u;  // the new node's level (select_level, operations.rs:76-83)
    for (uint32_t i = tid; i < ix.ds; i += nthreads) qs[i] = i < ix.dim ? __ldg(qg + i) : 0.f;
    {
      uint4* v4 = reinterpret_cast<uint4*>(vis);
      const uint32_t n16 = GLOBAL_VISITED ? (a.vis_words >> 2) : (a.lay.hash16 ? (hash_slots >> 3) : (hash_slots >> 2));
      const uint32_t fill = (GLOBAL_VISITED || a.lay.hash16) ? 0u : kInvalid;
      for (uint32_t i = tid; i < n16; i += nthreads) v4[i] = make_uint4(fill, fill, fill, fill);
    }
    team_sync<DIRECT>();
    if (METRIC == kCosine) t.qnorm = quad_dot(qs, qs, ix.dim, lane & 3);

    if (!DIRECT && warp != 0) {
      // ---- helper warps: serve distance requests until the leader is done with this query ----
      for (;;) {
        team_sync<DIRECT>();
        const uint32_t m = t.ctl[0];
        if (m == kDone) break;
        team_distances<METRIC, SQ8>(ix, t, m);
        team_sync<DIRECT>();
      }
      if (t.dbg && warp == 1 && lane == 0) {  // diagnostics: the first helper's share of the data path
        atomicAdd(a.dbg + 13, (unsigned long long)t.c_issue);
        atomicAdd(a.dbg + 14, (unsigned long long)t.c_wait);
        atomicAdd(a.dbg + 15, (unsigned long long)t.c_comp);
        t.c_issue = t.c_wait = t.c_comp = 0;
      }
      continue;
    }

    // ---- leader warp ----
    const long long q_t0 = t.dbg ? clock64() : 0;
    long long l0_t0 = 0;
    uint32_t c_sel = 0, c_adj = 0, c_req = 0, c_mrg = 0, c_vis = 0, n_hops = 0, n_spec = 0;
    t.c_issue = t.c_wait = t.c_comp = 0;
    uint32_t n_dist = 0, n_dist_upper = 0, n_expanded = 0, n_upper_hops = 0;
    uint32_t len = 0;
    bool overflow = false;

    if (ix.entry != kInvalid && ix.n != 0) {
      // entry distance (mod.rs:1129)
      uint32_t cur = ix.entry;
      if (lane == 0) cand_ids[0] = cur;
      float cur_d = __shfl_sync(kFullMask, request<METRIC, SQ8, DIRECT>(ix, t, 1), 0);
      n_dist = 1;
      n_dist_upper = 1;

      // greedy descent over levels max_level..1 (mod.rs:1134-1145, search.rs:259-309)
      // INSERT: only the levels above the new node's (insert_descent_phase, operations.rs:111-133)
      for (uint32_t level = ix.max_level; level >= (INSERT ? target + 1 : 1u); --level) {
        for (uint32_t it = 0; it < 1000; ++it) {
          const uint32_t lv = ix.levels[cur];
          const uint32_t ub = ix.up_base[cur];
          uint32_t nid = kInvalid;
          if (level <= lv && ub != kInvalid && lane < kUp)
            nid = __ldg(ix.up_adj + ((size_t)ub + level - 1) * kUp + lane);
          n_upper_hops += 1;
          const uint32_t m = __popc(__ballot_sync(kFullMask, nid != kInvalid));
          if (m == 0) break;
          if (lane < m) cand_ids[lane] = nid;
          const float d = request<METRIC, SQ8, DIRECT>(ix, t, m);
          n_dist += m;
          n_dist_upper += m;
          // arg-min, strict `<`, first stored neighbour wins ties (search.rs:272-277)
          float best = d;
          uint32_t bl = lane;
#pragma unroll
          for (uint32_t off = 16; off >= 1; off >>= 1) {
            const float od = __shfl_xor_sync(kFullMask, best, off);
            const uint32_t ol = __shfl_xor_sync(kFullMask, bl, off);
            if (od < best || (od == best && ol < bl)) {
              best = od;
              bl = ol;
            }
          }
          if (!(best < cur_d)) break;
          cur = __shfl_sync(kFullMask, nid, bl);
          cur_d = best;
        }
      }

      if (FILTERED) {
        // ---- beam_search_filtered (search.rs:352-398) ----
        // results R (visible nodes only, cap ef) = A/B lists; candidates = EVERY visited node: the closest
        // ones sit in the sorted window C/D (cap ef), the rest in the global overflow `ovf`.  Invariant:
        // max(window) <= o_min = min(overflow), so the window head is the global minimum; when the window
        // runs dry it is refilled with the smallest overflow entries.
        auto is_visible = [&](uint32_t id) { return ((a.visible[id >> 6] >> (id & 63)) & 1ull) != 0; };
        uint2* ovf = a.f_ovf + (size_t)blockIdx.x * a.f_ocap;
        uint32_t o_cnt = 0, c_head = 0, c_len = 1, r_len = 0, dummy = 0;
        float o_min = INFINITY;
        bool o_overflow = false;
        const bool entry_vis = is_visible(cur);
        if (lane == 0) {
          C_d[0] = cur_d;
          C_id[0] = cur;
          if (entry_vis) {
            A_d[0] = cur_d;
            A_id[0] = cur;
          }
        }
        r_len = entry_vis ? 1u : 0u;
        (void)visited_insert<GLOBAL_VISITED>(vis, cur, lane == 0, a.lay);
        uint32_t n_visited = 1;
        uint32_t spec_node = kInvalid, spec_nid = kInvalid;
        __syncwarp();
        for (;;) {
          if (c_head == c_len) {
            if (o_cnt == 0) break;
            // refill: stream the overflow through the window; what does not fit is compacted back in place
            const float worst_now = r_len ? A_d[r_len - 1] : INFINITY;
            const float drop = (r_len == ef) ? worst_now : INFINITY;
            const uint32_t total = o_cnt;
            uint32_t w = 0;
            o_min = INFINITY;
            c_head = 0;
            c_len = 0;
            for (uint32_t r = 0; r < total; r += 32) {
              const bool have = r + lane < total;
              const uint2 e = have ? ovf[r + lane] : make_uint2(0u, 0u);
              const float ed = __uint_as_float(e.x);
              __syncwarp();
              const bool el = have && !(ed > drop);
              c_len = rank_merge<true>(C_d, C_id, 0, c_len, D_d, D_id, ef, el, ed, e.y, tmp_ub, lane, &dummy, ovf, &w,
                                       a.f_ocap, &o_min, drop, &o_overflow);
              float* td = C_d; C_d = D_d; D_d = td;
              uint32_t* ti = C_id; C_id = D_id; D_id = ti;
            }
            o_cnt = w;
            if (c_len == 0) break;
          }
          const uint32_t c = C_id[c_head];
          const float cd = C_d[c_head];
          const float worst0 = r_len ? A_d[r_len - 1] : INFINITY;  // worst_result_distance(), search.rs:238-243
          if (cd > worst0) break;                                   // search.rs:374-376
          c_head += 1;
          n_expanded += 1;
          const uint32_t c2 = c_head < c_len ? C_id[c_head] : kInvalid;
          if (!GLOBAL_VISITED && n_visited + kL0 > hash_limit) {
            overflow = true;
            break;
          }
          const uint32_t nid = (c == spec_node) ? spec_nid : __ldg(ix.l0_adj + (size_t)c * kL0 + lane);
          if (c2 != kInvalid) {
            spec_node = c2;
            spec_nid = __ldg(ix.l0_adj + (size_t)c2 * kL0 + lane);
          } else {
            spec_node = kInvalid;
          }
          const uint32_t ins = visited_insert<GLOBAL_VISITED>(vis, nid, nid != kInvalid, a.lay);
          if (__any_sync(kFullMask, ins == 2u)) {
            overflow = true;
            break;
          }
          const bool isnew = ins == 1u;
          const uint32_t newmask = __ballot_sync(kFullMask, isnew);
          const uint32_t m = __popc(newmask);
          if (m == 0) continue;
          n_visited += m;
          if (isnew) cand_ids[__popc(newmask & ((1u << lane) - 1))] = nid;
          const float d = request<METRIC, SQ8, DIRECT>(ix, t, m);
          const uint32_t cid = lane < m ? cand_ids[lane] : kInvalid;
          n_dist += m;
          // results: visible && (d < worst || |R| < ef), search.rs:391-395 (batch form, see DESIGN.md §5)
          const bool vis_ok = lane < m && is_visible(cid);
          const bool r_elig = vis_ok && (r_len < ef || d < worst0);
          if (__any_sync(kFullMask, r_elig)) {
            r_len = rank_merge<false>(A_d, A_id, 0, r_len, B_d, B_id, ef, r_elig, d, cid, tmp_ub, lane, &dummy, nullptr,
                                      nullptr, 0, nullptr, INFINITY, nullptr);
            float* td = A_d; A_d = B_d; B_d = td;
            uint32_t* ti = A_id; A_id = B_id; B_id = ti;
          }
          // candidates: every new node (search.rs:389).  Once R is full `worst` only shrinks, so a candidate
          // beyond it can never pass the break test and is dropped.
          const float drop = (r_len == ef) ? A_d[r_len - 1] : INFINITY;
          const bool keep = lane < m && !(d > drop);
          const bool to_win = keep && d < o_min;
          const bool to_ovf = keep && !to_win;
          if (__any_sync(kFullMask, to_win) || c_head != 0) {
            c_len = rank_merge<true>(C_d, C_id, c_head, c_len, D_d, D_id, ef, to_win, d, cid, tmp_ub, lane, &dummy, ovf,
                                     &o_cnt, a.f_ocap, &o_min, drop, &o_overflow);
            c_head = 0;
            float* td = C_d; C_d = D_d; D_d = td;
            uint32_t* ti = C_id; C_id = D_id; D_id = ti;
          }
          const uint32_t omask = __ballot_sync(kFullMask, to_ovf);
          if (omask) {
            if (to_ovf) {
              const uint32_t o = o_cnt + __popc(omask & ((1u << lane) - 1));
              if (o < a.f_ocap) ovf[o] = make_uint2(__float_as_uint(d), cid);
              else o_overflow = true;
            }
            o_cnt += __popc(omask);
            float dm = to_ovf ? d : INFINITY;
#pragma unroll
            for (uint32_t off = 16; off >= 1; off >>= 1) dm = fminf(dm, __shfl_xor_sync(kFullMask, dm, off));
            o_min = fminf(o_min, dm);
            if (__any_sync(kFullMask, o_overflow)) o_overflow = true;
          }
          __syncwarp();
          if (o_overflow) break;
        }
        len = r_len;
        // candidate overflow buffer exhausted: the query is redone by the fallback pass, whose buffer holds every node
        if (o_overflow) {
          if (GLOBAL_VISITED) len = 0xFFFFFFFEu;  // cannot happen there (f_ocap == n)
          else overflow = true;
        }
      } else {
      // adjacency row of node c at level lvl, one id per lane (INVALID padded)
      auto adj_row = [&](uint32_t c, uint32_t lvl) -> uint32_t {
        if (!INSERT || lvl == 0) return __ldg(ix.l0_adj + (size_t)c * kL0 + lane);
        uint32_t nid = kInvalid;
        if (lane < kUp && lvl <= ix.levels[c]) nid = __ldg(ix.up_adj + ((size_t)ix.up_base[c] + lvl - 1) * kUp + lane);
        return nid;
      };
      // search(): one beam at level 0.  INSERT: insert_connection_phase (operations.rs:135-171) — one beam per level
      // target..0 with ef_construction, every one seeded with the SAME (cur, cur_d): the reference's second
      // finalize_results(1) drains an already empty heap, so the entry is never refined between levels; a level above
      // the current max_level yields just the old entry (one-way link, operations.rs:147).
      for (int32_t blevel = (int32_t)target; blevel >= 0 && !overflow; --blevel) {
      if (INSERT && blevel != (int32_t)target) {  // ctx.reset(): a fresh visited set per level
        uint4* v4 = reinterpret_cast<uint4*>(vis);
        const uint32_t n16 = GLOBAL_VISITED ? (a.vis_words >> 2) : (a.lay.hash16 ? (hash_slots >> 3) : (hash_slots >> 2));
        const uint32_t fill = (GLOBAL_VISITED || a.lay.hash16) ? 0u : kInvalid;
        for (uint32_t i = lane; i < n16; i += 32) v4[i] = make_uint4(fill, fill, fill, fill);
        __syncwarp();
      }
      // beam search (search.rs:311-350) on one sorted list
      if (lane == 0) {
        A_d[0] = cur_d;
        A_id[0] = cur;
      }
      (void)visited_insert<GLOBAL_VISITED>(vis, cur, lane == 0, a.lay);
      len = 1;
      uint32_t n_visited = 1;
      uint32_t row_node = kInvalid, row_nid = kInvalid;  // prefetched adjacency row of the runner-up
      // Speculation: while the helper warps gather hop h, the leader filters the runner-up's neighbours
      // through the visited set as if it were hop h+1.  If the merge confirms the runner-up (it does ~80 % of
      // the time) hop h+1 starts with its request ready; otherwise the keys are taken back (visited_undo),
      // which restores the table exactly, and the hop proceeds as usual.  Results and counters are unchanged.
      bool sp_valid = false, sp_inserted = false;
      uint32_t sp_node = kInvalid, sp_where = 0, sp_m = 0;
      uint32_t scan_from = 0;                               // list entries below this index are expanded
      __syncwarp();
      if (t.dbg) l0_t0 = clock64();

      for (;;) {
        const long long h0 = t.dbg ? clock64() : 0;
        // closest unexpanded entry == the reference's candidates.pop() that passes `d <= worst`;
        // the runner-up is the likely next hop.
        // Everything below `scan_from` is known to be expanded, so one 32-wide probe usually suffices.
        uint32_t idx = 0xFFFFFFFFu, idx2 = 0xFFFFFFFFu;
        for (uint32_t base = scan_from; base < len; base += 32) {
          const uint32_t i = base + lane;
          uint32_t um = __ballot_sync(kFullMask, i < len && !(A_id[i] & kExpandedBit));
          if (um) {
            idx = base + __ffs(um) - 1;
            um &= um - 1;
            if (um) idx2 = base + __ffs(um) - 1;
            break;
          }
        }
        if (idx >= len) break;
        const uint32_t c = A_id[idx];
        const uint32_t c2 = idx2 < len ? A_id[idx2] : kInvalid;
        __syncwarp();
        if (lane == 0) A_id[idx] = c | kExpandedBit;
        __syncwarp();
        n_expanded += 1;
        scan_from = idx + 1;
        const long long h1 = t.dbg ? clock64() : 0;

        const bool hit = sp_valid && sp_node == c;
        if (sp_valid && !hit) visited_undo<GLOBAL_VISITED>(vis, sp_inserted, sp_where, a.lay);
        sp_valid = false;
        uint32_t m;
        if (hit) {
          // c's unvisited neighbours are already in the table; their ids wait in cand_next (stored order)
          if (t.dbg) n_spec += 1;
          m = sp_m;
          if (lane < m) cand_ids[lane] = cand_next[lane];
          if (c2 != kInvalid) {
            row_node = c2;
            row_nid = adj_row(c2, (uint32_t)blevel);
          } else {
            row_node = kInvalid;
          }
          if (m == 0) continue;
        } else {
          if (!GLOBAL_VISITED && n_visited + kL0 > hash_limit) {
            overflow = true;
            break;
          }
          const uint32_t nid = (c == row_node) ? row_nid : adj_row(c, (uint32_t)blevel);
          if (c2 != kInvalid) {
            row_node = c2;
            row_nid = adj_row(c2, (uint32_t)blevel);
          } else {
            row_node = kInvalid;
          }
          const long long v0 = t.dbg ? clock64() : 0;
          const uint32_t ins = visited_insert<GLOBAL_VISITED>(vis, nid, nid != kInvalid, a.lay);
          if (t.dbg) c_vis += (uint32_t)(clock64() - v0);
          if (__any_sync(kFullMask, ins == 2u)) {
            overflow = true;
            break;
          }
          const bool isnew = ins == 1u;
          const uint32_t newmask = __ballot_sync(kFullMask, isnew);
          m = __popc(newmask);
          if (m == 0) continue;
          // compact to slots 0..m-1 in stored order
          if (isnew) cand_ids[__popc(newmask & ((1u << lane) - 1))] = nid;
        }
        n_visited += m;
        const long long h2 = t.dbg ? clock64() : 0;
        const float d = request<METRIC, SQ8, DIRECT>(ix, t, m, [&] {
          // hop h+1 prepared under hop h's gather (leader only; cand_ids belongs to the helpers meanwhile)
          if (row_node == kInvalid) return;
          if (!GLOBAL_VISITED && n_visited + kL0 > hash_limit) return;  // the real hop reports the overflow
          uint32_t w = 0;
          const uint32_t ins2 = visited_insert<GLOBAL_VISITED>(vis, row_nid, row_nid != kInvalid, a.lay, &w);
          sp_inserted = ins2 == 1u;
          sp_where = w;
          if (__any_sync(kFullMask, ins2 == 2u)) {
            visited_undo<GLOBAL_VISITED>(vis, sp_inserted, sp_where, a.lay);
            return;
          }
          const uint32_t nm = __ballot_sync(kFullMask, sp_inserted);
          sp_m = __popc(nm);
          if (sp_inserted) cand_next[__popc(nm & ((1u << lane) - 1))] = row_nid;
          sp_node = row_node;
          sp_valid = true;
        });
        const long long h3 = t.dbg ? clock64() : 0;
        if (t.dbg) {
          c_sel += (uint32_t)(h1 - h0);
          c_adj += (uint32_t)(h2 - h1);
          c_req += (uint32_t)(h3 - h2);
          n_hops += 1;
        }
        const uint32_t cid = lane < m ? cand_ids[lane] : kInvalid;
        n_dist += m;

        // admission (search.rs:344): d < worst || results.len() < ef, applied to the batch
        const float worst = (len == ef) ? A_d[len - 1] : INFINITY;
        const bool elig = (lane < m) && (len < ef || d < worst);
        const uint32_t emask = __ballot_sync(kFullMask, elig);
        const uint32_t mp = __popc(emask);
        if (mp == 0) continue;

        // insertion point among old entries: old entries win ties (they were admitted first)
        uint32_t ub = 0;
        if (elig) {
          uint32_t lo = 0, hi = len;
          while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (A_d[mid] <= d) lo = mid + 1;
            else hi = mid;
          }
          ub = lo;
          tmp_ub[__popc(emask & ((1u << lane) - 1))] = ub;
        }
        // rank among the new entries: (distance, stored order)
        uint32_t rank = 0;
        for (uint32_t e = emask; e; e &= e - 1) {
          const uint32_t bsrc = __ffs(e) - 1;
          const float db = __shfl_sync(kFullMask, d, bsrc);
          rank += (db < d || (db == d && bsrc < lane)) ? 1u : 0u;
        }
        __syncwarp();
        // in place, from the top down in batches of kMergeBatch 32-entry blocks: a batch is read into registers, the
        // warp synchronises, the batch is written at its shifted positions (always >= the old ones, and the
        // batches above have already moved), the warp synchronises
        for (int32_t top = (int32_t)((len - 1) >> 5); top >= 0; top -= kMergeBatch) {
          float od[kMergeBatch];
          uint32_t oi[kMergeBatch], np[kMergeBatch];
#pragma unroll
          for (int u = 0; u < kMergeBatch; ++u) {
            const int32_t blk = top - u;
            const uint32_t i = (uint32_t)blk * 32 + lane;
            np[u] = 0xFFFFFFFFu;
            od[u] = 0.f;
            oi[u] = 0;
            if (blk >= 0 && i < len) {
              od[u] = A_d[i];
              oi[u] = A_id[i];
              np[u] = i;
            }
          }
          for (uint32_t j = 0; j < mp; ++j) {
            const uint32_t tv = tmp_ub[j];
#pragma unroll
            for (int u = 0; u < kMergeBatch; ++u) np[u] += (np[u] != 0xFFFFFFFFu && tv <= (uint32_t)(top - u) * 32 + lane) ? 1u : 0u;
          }
          __syncwarp();
#pragma unroll
          for (int u = 0; u < kMergeBatch; ++u)
            if (np[u] < ef) {
              A_d[np[u]] = od[u];
              A_id[np[u]] = oi[u];
            }
          __syncwarp();
        }
        uint32_t my_np = 0xFFFFFFFFu;
        if (elig) {
          const uint32_t np = ub + rank;
          if (np < ef) {
            A_d[np] = d;
            A_id[np] = cid;
            my_np = np;
          }
        }
        scan_from = min(scan_from, __reduce_min_sync(kFullMask, my_np));
        len = min(len + mp, ef);
        __syncwarp();
        if (t.dbg) c_mrg += (uint32_t)(clock64() - h3);
      }
      if (INSERT && !overflow) {
        // the level's selection: the beam's nearest m0 (level 0) / m results in ascending order (operations.rs:157-162)
        const uint32_t cnt = min(len, blevel == 0 ? a.ins_m0 : a.ins_m);
        uint32_t* os = a.ins_sel + ((size_t)qi * kInsLevels + (uint32_t)blevel) * kInsSelMax;
        for (uint32_t i = lane; i < cnt; i += 32) os[i] = A_id[i] & ~kExpandedBit;
        if (lane == 0) a.ins_cnt[(size_t)qi * kInsLevels + (uint32_t)blevel] = (uint8_t)cnt;
        __syncwarp();
      }
      }  // levels
      }  // !FILTERED
    }
    if (t.dbg && lane == 0) {
      const long long q_t1 = clock64();
      atomicAdd(a.dbg + 0, (unsigned long long)n_hops);
      atomicAdd(a.dbg + 1, (unsigned long long)c_sel);
      atomicAdd(a.dbg + 2, (unsigned long long)c_adj);
      atomicAdd(a.dbg + 3, (unsigned long long)c_req);
      atomicAdd(a.dbg + 4, (unsigned long long)c_mrg);
      atomicAdd(a.dbg + 5, (unsigned long long)t.c_wait);
      atomicAdd(a.dbg + 6, (unsigned long long)t.c_issue);
      atomicAdd(a.dbg + 7, (unsigned long long)t.c_comp);
      atomicAdd(a.dbg + 8, (unsigned long long)n_spec);
      atomicAdd(a.dbg + 9, (unsigned long long)(q_t1 - q_t0));
      atomicAdd(a.dbg + 10, (unsigned long long)(l0_t0 - q_t0));
      atomicAdd(a.dbg + 11, 1ull);
      atomicAdd(a.dbg + 12, (unsigned long long)c_vis);
    }

    // release the helper warps
    if (lane == 0) t.ctl[0] = kDone;
    team_sync<DIRECT>();

    if (overflow) {
      // shared visited table cannot take more keys: hand the query to the global-bitset pass (exact, rare)
      if (lane == 0) a.overflow_list[atomicAdd(a.overflow_count, 1u)] = qi;
      continue;
    }
    if (INSERT) continue;  // the per-level selections are the output

    // ---- finalize_results(k) (search.rs:245-252) + SearchResult mapping (mod.rs:1159-1171) ----
    const bool f_fail = FILTERED && len == 0xFFFFFFFEu;
    if (f_fail) len = 0;
    const uint32_t count = min(len, a.k);
    for (uint32_t i = lane; i < a.k; i += 32) {
      const size_t o = (size_t)qi * a.k + i;
      if (i < count) {
        const uint32_t id = A_id[i] & ~kExpandedBit;
        a.out_row_ids[o] = ix.row_ids[id];
        if (a.out_node_ids) a.out_node_ids[o] = id;
        a.out_dist[o] = A_d[i];
      } else {
        a.out_row_ids[o] = 0xFFFFFFFFFFFFFFFFull;
        if (a.out_node_ids) a.out_node_ids[o] = kInvalid;
        a.out_dist[o] = INFINITY;
      }
    }
    if (lane == 0) {
      if (a.tstats) {
        atomicMax(&a.tstats->vis_max, n_dist - n_dist_upper + 1);
        atomicAdd(&a.tstats->sum_dist, (unsigned long long)(n_dist - n_dist_upper));
        atomicAdd(&a.tstats->sum_exp, (unsigned long long)n_expanded);
      }
      a.out_counts[qi] = f_fail ? 0xFFFFFFFEu : count;
      if (a.out_stats) {
        uint32_t* s = a.out_stats + (size_t)qi * 4;
        s[0] = n_dist;
        s[1] = n_dist_upper;
        s[2] = n_expanded;
        s[3] = n_upper_hops;
      }
    }
  }
}

// staged form: a team of 2-4 warps per query, rows through shared-memory staging (TMA bulk copies)
template <int METRIC, bool GLOBAL_VISITED, bool FILTERED, bool SQ8 = false>
__global__ void __launch_bounds__(128, TURDB_MIN_CTAS) hnsw_search_kernel(const SearchArgs a) {
  hnsw_search_body<METRIC, GLOBAL_VISITED, FILTERED, SQ8, false>(a);
}

// direct form: one warp per query, rows straight into registers (short rows)
#ifndef TURDB_WARP_MIN_CTAS
#define TURDB_WARP_MIN_CTAS 20
#endif
template <int METRIC, bool GLOBAL_VISITED, bool FILTERED>
__global__ void __launch_bounds__(32, TURDB_WARP_MIN_CTAS) hnsw_search_warp_kernel(const SearchArgs a) {
  hnsw_search_body<METRIC, GLOBAL_VISITED, FILTERED, false, true>(a);
}

// The insert path's searches (insert_with_callback, mod.rs:999-1084: greedy descent, then one ef_construction beam per
// level of the new node), always squared L2 (mod.rs:1031,1046), staged and direct form.
template <bool GLOBAL_VISITED>
__global__ void __launch_bounds__(128, TURDB_MIN_CTAS) hnsw_insert_search_kernel(const SearchArgs a) {
  hnsw_search_body<kL2, GLOBAL_VISITED, false, false, false, true>(a);
}
template <bool GLOBAL_VISITED>
__global__ void __launch_bounds__(32, TURDB_WARP_MIN_CTAS) hnsw_insert_search_warp_kernel(const SearchArgs a) {
  hnsw_search_body<kL2, GLOBAL_VISITED, false, false, true, true>(a);
}

}  // namespace turdb
