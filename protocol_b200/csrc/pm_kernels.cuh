// pm_kernels.cuh — sm_100a kernels of the matching pass.
//
//   pm_build_cost   cost-matrix build: int64 cost[t][w] for a tile of asks x a
//                   stripe of workers, HBM-write-bound (8 B per evaluation);
//                   pm_build_cost_fast<.., uint16_t> writes 16-bit price words
//                   (2 B per evaluation) when every worker price is <= 0xFFFE
//   pm_argmin       one read of the tile (8 B per evaluation): per-ask packed
//                   (min_cost, argmin) + feasible count, per-worker first ask;
//                   pm_argmin16 the same from a 16-bit tile (2 B per evaluation)
//   pm_fused_eval   the same outputs without materialising the matrix
//   pm_hist / pm_check_tails / pm_sweep / pm_emit_* : resolution sweep that turns
//                   "first feasible ask per worker" into the reference's groups
//
// Reference semantics being reproduced: NodeGroupsPlugin::try_form_new_groups,
// crates/orchestrator/src/plugins/node_groups/mod.rs:478-628.
#pragma once
#include "pm_device.cuh"

namespace pm {

struct EvalParams {
  const uint4* __restrict__ wa;       // plane A [n_workers]
  const uint4* __restrict__ wb;       // plane B [n_workers]
  const DevAsk* __restrict__ asks;    // [n_asks] priority order
  const DevOpt* __restrict__ opts;    // CSR, ask order
  const DevOptF* __restrict__ opts_fast;  // same CSR, fast-path form
  const FastRow* __restrict__ frows;      // [n_asks] fast build kernel's view of an ask (first option inline)
  const uint32_t* __restrict__ bits;  // [(n_patterns+1) * words], row 0 all-ones
  const uint32_t* __restrict__ nacc;  // worker-major acceptance (pm_worker_nacc), or null: per worker the mask of the pattern
                                      // rows that REJECT its model.  Then `bits` is the one-word table word[r] = ~(1 << r) and a
                                      // worker's mmask is nacc[w]: the fast clause ~word & mmask = (1 << r) & nacc[w] is the same
                                      // test with the roles of row and worker swapped — no table lookup per (row, worker) pair,
                                      // however many distinct model strings the pool has (at most 30 patterns)
  uint32_t words;
  uint32_t n_workers;                 // global
  uint32_t n_asks;
  uint32_t n_opts;
  uint32_t n_bits_rows;               // n_patterns + 1
  uint32_t sign_shift;                // always 31.  A run-time value on purpose: with a literal shift ptxas proves the
                                      // result is 0/1 and turns the two multiply-adds that form the packed cost back
                                      // into a compare and two selects on the (busier) ALU pipe
};

// ------------------------------------------------------------------ evaluation core
constexpr int kEvalThreads = 256;
constexpr int kEvalWPT = 4;                          // workers per thread: two 16 B stores per row
constexpr int kEvalCols = kEvalThreads * kEvalWPT;   // 1024 workers per CTA stripe
constexpr int kEvalRows = 128;                       // asks per CTA (staged in shared memory)
constexpr int kOptCap = 384;                         // options staged at a time
constexpr int kBitsCap = 2048;                       // acceptance-table words kept in shared memory

struct __align__(128) EvalStage {
  DevAsk ask[kEvalRows];
  DevOpt opt[kOptCap];
  uint32_t bits[kBitsCap];
  uint64_t bar;
};

// The predicate for one staged ask against WPT register-resident workers, as
// all-ones / zero masks.  Ask and option operands are warp-uniform shared-memory
// reads; each clause is one subtract/and plus one ISETP chained on a single
// predicate (inline PTX keeps ptxas from materialising booleans in registers).
__device__ __forceinline__ uint32_t base_mask(const DevAsk& a, const WorkerReg& w) {
  uint32_t r;
  asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\t"
      "and.b32 t, %1, %2;\n\t"
      "setp.eq.u32 p, t, %2;\n\t"
      "setp.ge.and.u32 p, %3, %4, p;\n\t"
      "setp.ge.and.u32 p, %5, %6, p;\n\t"
      "setp.ge.and.u32 p, %7, %8, p;\n\t"
      "selp.b32 %0, -1, 0, p;\n\t}"
      : "=r"(r)
      : "r"(w.flags), "r"(a.need), "r"(w.cores), "r"(a.cpu_cores), "r"(w.ram), "r"(a.ram_mb),
        "r"(w.storage), "r"(a.storage_gb));
  return r;
}

// GpuSpecs::meets for one option (node.rs:443-527).  `word` is the worker's word
// of the option's acceptance row (row 0 is all-ones: no model clause).
__device__ __forceinline__ uint32_t opt_mask(const DevOpt& q, const WorkerReg& w, uint32_t word) {
  uint32_t r;
  asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\t"
      "and.b32 t, %1, %2;\n\t"
      "setp.eq.u32 p, t, %2;\n\t"            // presence bits
      "and.b32 t, %3, %4;\n\t"
      "setp.eq.and.u32 p, t, %5, p;\n\t"     // count == (or unconstrained)
      "sub.u32 t, %6, %7;\n\t"
      "setp.le.and.u32 p, t, %8, p;\n\t"     // memory_mb in [lo, hi]
      "sub.u32 t, %9, %11;\n\t"
      "and.b32 t, t, %10;\n\t"               // workers without count*memory skip the clause
      "setp.le.and.u32 p, t, %12, p;\n\t"    // count * memory_mb in [lo, hi]
      "and.b32 t, %13, %14;\n\t"
      "setp.ne.and.u32 p, t, 0, p;\n\t"      // model accepted
      "selp.b32 %0, -1, 0, p;\n\t}"
      : "=r"(r)
      : "r"(w.flags), "r"(q.need), "r"(w.count_eff), "r"(q.count_mask), "r"(q.count),
        "r"(w.mem_eff), "r"(q.mem_lo), "r"(q.mem_span), "r"(w.tot), "r"(w.tot_keep), "r"(q.tot_lo),
        "r"(q.tot_span), "r"(word), "r"(w.mmask));
  return r;
}

// BITS: 0 = acceptance table in global memory, 1 = in shared memory, 2 = in shared
// memory with one word per row (<= 32 worker models): the word is warp-uniform.
template <int WPT, int BITS>
__device__ __forceinline__ void eval_row(const EvalStage& s, const DevAsk& a, uint32_t obegin,
                                         const WorkerReg (&w)[WPT],
                                         const uint32_t* __restrict__ gbits, uint32_t words,
                                         uint32_t (&f)[WPT]) {
#pragma unroll
  for (int k = 0; k < WPT; ++k) f[k] = base_mask(a, w[k]);
  if (a.n_opts != 0u) {
    uint32_t any[WPT];
#pragma unroll
    for (int k = 0; k < WPT; ++k) any[k] = 0u;
    const uint32_t o0 = a.opt_off - obegin;
    for (uint32_t o = 0; o < a.n_opts; ++o) {
      const DevOpt q = s.opt[o0 + o];
      if (BITS == 2) {
        const uint32_t word = s.bits[q.pattern_row];
#pragma unroll
        for (int k = 0; k < WPT; ++k) any[k] |= opt_mask(q, w[k], word);
      } else {
        const uint32_t rowoff = q.pattern_row * words;
#pragma unroll
        for (int k = 0; k < WPT; ++k) {
          const uint32_t word = (BITS == 1) ? s.bits[rowoff + w[k].mword] : __ldg(gbits + rowoff + w[k].mword);
          any[k] |= opt_mask(q, w[k], word);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < WPT; ++k) f[k] &= any[k];
  }
}

// Fast path (all operands < 2^31, counts < 2^16; layout and derivation at DevOptF in pm_device.cuh): the SIGN BIT of
// fail[k] is set <=> worker k does not meet the ask.  Per worker and option: 5 LOP3 on the ALU pipe, 7 IMAD-pipe
// adds/subtractions; clauses are never compared, only OR-ed (AND across the ask's OR-options).  Every converted ask
// has at least one option row (pm_ask_convert adds a neutral one), so there is no option-less special case.
template <int WPT, int BITS>
__device__ __forceinline__ void eval_opt_fast(const EvalStage& s, const DevOptF& q, const WorkerReg (&w)[WPT],
                                              const uint32_t* __restrict__ gbits, uint32_t words, uint32_t (&u)[WPT]) {
  const uint32_t rowoff = q.pattern_row * words;
  const uint32_t uword = (BITS == 2) ? s.bits[q.pattern_row] : 0u;
#pragma unroll
  for (int k = 0; k < WPT; ++k) {
    const uint32_t word = (BITS == 2) ? uword
                          : (BITS == 1) ? s.bits[rowoff + w[k].mword] : __ldg(gbits + rowoff + w[k].mword);
    const uint32_t z = ((w[k].key & q.m) ^ q.v) | (~word & w[k].mmask);          // < 2^31, non-zero = fails
    const uint32_t r = (w[k].mem_eff - q.mem_lo) | (q.mem_hi - w[k].mem_eff) |
                       (((w[k].tot - q.tot_lo) | (q.tot_hi - w[k].tot)) & w[k].tot_keep);
    u[k] = (0u - z) | r;    // z < 2^31: the negation has its sign set exactly when z != 0
  }
}

template <int WPT, int BITS>
__device__ __forceinline__ void eval_row_fast(const EvalStage& s, const DevAsk& a, uint32_t obegin,
                                              const WorkerReg (&w)[WPT],
                                              const uint32_t* __restrict__ gbits, uint32_t words,
                                              uint32_t (&fail)[WPT]) {
  const DevOptF* optf = reinterpret_cast<const DevOptF*>(s.opt) + (a.opt_off - obegin);
  uint32_t um[WPT];
  eval_opt_fast<WPT, BITS>(s, optf[0], w, gbits, words, um);
  for (uint32_t o = 1; o < a.n_opts; ++o) {   // OR-options (node.rs:420-438): the ask fails only if every option does
    uint32_t u[WPT];
    eval_opt_fast<WPT, BITS>(s, optf[o], w, gbits, words, u);
#pragma unroll
    for (int k = 0; k < WPT; ++k) um[k] &= u[k];
  }
#pragma unroll
  for (int k = 0; k < WPT; ++k)
    fail[k] = um[k] | (w[k].cores - a.cpu_cores) | (w[k].ram - a.ram_mb) | (w[k].storage - a.storage_gb);
}

// Slow path for an ask whose option list alone exceeds the staging capacity.
template <int WPT>
__device__ __noinline__ void eval_row_global(const EvalParams& p, const DevAsk& a,
                                             const WorkerReg (&w)[WPT], uint32_t (&f)[WPT]) {
#pragma unroll
  for (int k = 0; k < WPT; ++k) f[k] = ask_meets(a, p.opts, w[k], p.bits, p.words) ? 0xFFFFFFFFu : 0u;
}

template <int WPT>
__device__ __forceinline__ void load_workers(const EvalParams& p, uint32_t w0, uint32_t nw,
                                             uint32_t c, WorkerReg (&w)[WPT]) {
#pragma unroll
  for (int k = 0; k < WPT; ++k) {
    const uint32_t col = c + k;
    if (col < nw) {
      w[k] = make_worker(__ldg(p.wa + w0 + col), __ldg(p.wb + w0 + col));
      if (p.nacc) w[k].mmask = __ldg(p.nacc + w0 + col);
    } else w[k] = null_worker();
  }
}

// Drives `body(row_in_tile, ask, obegin, staged)` over rows [r0, r1) of the tile:
// ask headers, then as many option rows as fit, arrive in shared memory through
// 1-D TMA bulk copies signalled on one mbarrier.
template <class Body>
__device__ __forceinline__ void for_each_staged_row(EvalStage& s, const EvalParams& p, bool fast,
                                                    uint32_t t0, uint32_t r0, uint32_t r1, Body&& body) {
  const DevOpt* opt_src = fast ? reinterpret_cast<const DevOpt*>(p.opts_fast) : p.opts;
  if (threadIdx.x == 0) mbar_init(&s.bar, 1);
  const uint32_t total_words = (p.n_bits_rows)*p.words;
  if (total_words <= (uint32_t)kBitsCap)
    for (uint32_t i = threadIdx.x; i < total_words; i += blockDim.x) s.bits[i] = __ldg(p.bits + i);
  __syncthreads();
  uint32_t phase = 0;
  const uint32_t nrows = r1 - r0;
  if (threadIdx.x == 0) {
    mbar_expect_tx(&s.bar, nrows * (uint32_t)sizeof(DevAsk));
    bulk_g2s(s.ask, p.asks + t0 + r0, nrows * (uint32_t)sizeof(DevAsk), &s.bar);
  }
  mbar_wait(&s.bar, phase);
  phase ^= 1u;
  uint32_t row = 0;
  while (row < nrows) {
    const uint32_t obegin = s.ask[row].opt_off;
    // rows [row, row+n) whose options fit (option offsets are non-decreasing in ask order)
    const uint32_t r = row + threadIdx.x;
    const bool fits = r < nrows && (s.ask[r].opt_off + s.ask[r].n_opts - obegin) <= (uint32_t)kOptCap;
    const uint32_t n = (uint32_t)__syncthreads_count(fits);
    if (n == 0) {  // one ask with more options than the stage holds
      body(row, s.ask[row], 0u, false);
      ++row;
      continue;
    }
    const uint32_t oend = s.ask[row + n - 1].opt_off + s.ask[row + n - 1].n_opts;
    if (oend > obegin) {
      if (threadIdx.x == 0) {
        mbar_expect_tx(&s.bar, (oend - obegin) * (uint32_t)sizeof(DevOpt));
        bulk_g2s(s.opt, opt_src + obegin, (oend - obegin) * (uint32_t)sizeof(DevOpt), &s.bar);
      }
      mbar_wait(&s.bar, phase);
      phase ^= 1u;
    }
    for (uint32_t i = 0; i < n; ++i) body(row + i, s.ask[row + i], obegin, true);
    row += n;
    if (row < nrows) __syncthreads();  // everyone is done with s.opt before it is overwritten
  }
}

// ------------------------------------------------------------------ build
// grid = (ld / 1024, ceil(nt / 128)); each thread owns 4 workers in registers and walks
// the staged asks, emitting two 128-bit streaming stores per row: a warp writes 1 KB
// contiguous (two fully coalesced 512-byte stores), the CTA 8 KB contiguous per row.
// ld is a multiple of the CTA's 1024 columns (columns past the shard hold the "infeasible" pattern of a null
// worker), so the stores need no bounds test.  Fast form: the packed cost is formed from the predicate's sign bit
// with one shift and two multiply-adds per worker — no compare, no select (see DevOptF).
template <int BITS, bool FAST, int MINB = 2>
__global__ void __launch_bounds__(kEvalThreads, MINB)
pm_build_cost(EvalParams p, uint32_t t0, uint32_t nt, uint32_t w0, uint32_t nw,
              long long* __restrict__ cost, size_t ld) {
  __shared__ EvalStage s;
  const uint32_t r0 = blockIdx.y * kEvalRows;
  const uint32_t r1 = min(nt, r0 + (uint32_t)kEvalRows);
  // A warp owns 128 consecutive columns; a lane owns the pairs (2l, 2l+1) and (64+2l, 64+2l+1), so each of
  // its two 128-bit stores per row is part of a fully coalesced 512-byte warp store (4 whole lines).
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t cbase = blockIdx.x * kEvalCols + (threadIdx.x >> 5) * 128u + lane * 2u;
  WorkerReg w[kEvalWPT];
  uint32_t gw[kEvalWPT], dx[kEvalWPT], dy[kEvalWPT];
#pragma unroll
  for (int k = 0; k < kEvalWPT; ++k) {
    const uint32_t col = cbase + (k >> 1) * 64u + (k & 1);
    gw[k] = w0 + col;
    if (col < nw) {
      w[k] = make_worker(__ldg(p.wa + w0 + col), __ldg(p.wb + w0 + col));
      if (p.nacc) w[k].mmask = __ldg(p.nacc + w0 + col);
    } else w[k] = null_worker();
    dx[k] = 0xFFFFFFFFu - gw[k];          // infeasible: 0x7FFFFFFF_FFFFFFFF = feasible word + (0/1) * difference
    dy[k] = 0x7FFFFFFFu - w[k].price;
  }
  uint4* out = reinterpret_cast<uint4*>(cost + (size_t)r0 * ld + cbase);
  const size_t row_stride = ld / 2;   // in 16-byte units; rows are visited in increasing order
  for_each_staged_row(s, p, FAST, t0, r0, r1, [&](uint32_t, const DevAsk& a, uint32_t obegin, bool staged) {
    uint4 v0, v1;
    // feasible: (price << 32) | worker ; infeasible: 0x7FFFFFFF_FFFFFFFF
    if (FAST && staged) {
      uint32_t fail[kEvalWPT];
      eval_row_fast<kEvalWPT, BITS>(s, a, obegin, w, p.bits, p.words, fail);
      const uint32_t sh = p.sign_shift;
      const uint32_t b0 = fail[0] >> sh, b1 = fail[1] >> sh, b2 = fail[2] >> sh, b3 = fail[3] >> sh;
      v0.x = b0 * dx[0] + gw[0]; v0.y = b0 * dy[0] + w[0].price;
      v0.z = b1 * dx[1] + gw[1]; v0.w = b1 * dy[1] + w[1].price;
      v1.x = b2 * dx[2] + gw[2]; v1.y = b2 * dy[2] + w[2].price;
      v1.z = b3 * dx[3] + gw[3]; v1.w = b3 * dy[3] + w[3].price;
    } else {
      uint32_t f[kEvalWPT];
      if (staged) eval_row<kEvalWPT, BITS>(s, a, obegin, w, p.bits, p.words, f);
      else eval_row_global<kEvalWPT>(p, a, w, f);
      v0.x = gw[0] | ~f[0]; v0.y = (w[0].price & f[0]) | (0x7FFFFFFFu & ~f[0]);
      v0.z = gw[1] | ~f[1]; v0.w = (w[1].price & f[1]) | (0x7FFFFFFFu & ~f[1]);
      v1.x = gw[2] | ~f[2]; v1.y = (w[2].price & f[2]) | (0x7FFFFFFFu & ~f[2]);
      v1.z = gw[3] | ~f[3]; v1.w = (w[3].price & f[3]) | (0x7FFFFFFFu & ~f[3]);
    }
    __stcs(out, v0);
    __stcs(out + 32, v1);     // + 64 columns
    out += row_stride;
  });
}

// ------------------------------------------------------------------ build, fast form
// Same decomposition and output as pm_build_cost, for tables that fit the fast predicate.  What changed after the
// round-2 profile (profiles/r02_summary.md: ALU pipe no longer the limiter, warps waiting on chained shared-memory
// loads — ask -> its option -> the option's acceptance word — and on the previous row's store reading its registers):
//   * one FastRow per ask: everything a single-option ask needs in three 128-bit loads whose address depends only on
//     the row number; the rows of the CTA arrive by ONE 1-D TMA bulk copy;
//   * the next row's FastRow is loaded while the current row is evaluated (explicit double buffer in registers);
//   * further OR-options (one ask in ten) are read straight from global memory, warp-uniform and L1-resident.
template <int WPT, int BITS>
__device__ __forceinline__ void eval_fast_first(const FastRow& q, const uint32_t* sbits, const WorkerReg (&w)[WPT],
                                                const uint32_t* __restrict__ gbits, uint32_t words, uint32_t (&u)[WPT]) {
#pragma unroll
  for (int k = 0; k < WPT; ++k) {
    const uint32_t word = (BITS == 2) ? q.wp
                          : (BITS == 1) ? sbits[q.wp * words + w[k].mword] : __ldg(gbits + q.wp * words + w[k].mword);
    const uint32_t z = ((w[k].key & q.m) ^ q.v) | (~word & w[k].mmask);
    const uint32_t r = (w[k].mem_eff - q.mem_lo) | (q.mem_hi - w[k].mem_eff) |
                       (((w[k].tot - q.tot_lo) | (q.tot_hi - w[k].tot)) & w[k].tot_keep);
    u[k] = (0u - z) | r;
  }
}

template <int WPT, int BITS>
__device__ __forceinline__ void eval_fast_more(const DevOptF* __restrict__ gopts, uint32_t n_more, const uint32_t* sbits,
                                               const WorkerReg (&w)[WPT], const uint32_t* __restrict__ gbits,
                                               uint32_t words, uint32_t (&um)[WPT]) {
  for (uint32_t o = 0; o < n_more; ++o) {
    const uint4 q0 = __ldg(reinterpret_cast<const uint4*>(gopts + o));
    const uint4 q1 = __ldg(reinterpret_cast<const uint4*>(gopts + o) + 1);   // {tot_lo, tot_hi, pattern_row, pad}
    const uint32_t uword = (BITS == 2) ? __ldg(gbits + q1.z) : 0u;
#pragma unroll
    for (int k = 0; k < WPT; ++k) {
      const uint32_t word = (BITS == 2) ? uword
                            : (BITS == 1) ? sbits[q1.z * words + w[k].mword] : __ldg(gbits + q1.z * words + w[k].mword);
      const uint32_t z = ((w[k].key & q0.x) ^ q0.y) | (~word & w[k].mmask);
      const uint32_t r = (w[k].mem_eff - q0.z) | (q0.w - w[k].mem_eff) |
                         (((w[k].tot - q1.x) | (q1.y - w[k].tot)) & w[k].tot_keep);
      um[k] &= (0u - z) | r;
    }
  }
}

template <int ROWS>
struct __align__(128) FastStage {
  FastRow row[ROWS];
  uint32_t bits[kBitsCap];
  uint64_t bar;
};
constexpr int kFastRows = 512;   // asks per CTA: the prologue (worker rows from L2, the TMA of the FastRows) is paid once per CTA
                                 // (measured on cfg3: 128 rows 119.1 ms/step, 256 rows 116.3, 512 rows 113.8 — profiles/r02_build_rows.txt)

// Word = long long: the int64 packed cost (price << 32 | worker, 0x7FFFFFFF_FFFFFFFF when infeasible), 8 B per
// evaluation; a lane owns the column pairs (2l, 2l+1) and (64+2l, 64+2l+1) of its warp's 128 columns (two 128-bit stores
// per row).  Word = uint16_t: the price word (price, 0xFFFF when infeasible), 2 B per evaluation, for worker tables whose
// prices are all <= 0xFFFE — the worker index is the column, so the word carries everything the argmin needs; a lane
// owns 4 consecutive columns and writes them with one 64-bit store per row (a warp 256 B contiguous).
template <int BITS, int ROWS = kFastRows, typename Word = long long, int MINB = 2>
__global__ void __launch_bounds__(kEvalThreads, MINB)
pm_build_cost_fast(EvalParams p, uint32_t t0, uint32_t nt, uint32_t w0, uint32_t nw, Word* __restrict__ cost, size_t ld) {
  static_assert(sizeof(Word) == 2 || sizeof(Word) == 8, "cost word is int64 or 16-bit");
  if constexpr (sizeof(Word) == 2) {
    __shared__ FastStage<ROWS> s;
    const uint32_t r0 = blockIdx.y * ROWS;
    const uint32_t nrows = min(nt - r0, (uint32_t)ROWS);
    if (threadIdx.x == 0) {
      mbar_init(&s.bar, 1);
      mbar_expect_tx(&s.bar, nrows * (uint32_t)sizeof(FastRow));
      bulk_g2s(s.row, p.frows + t0 + r0, nrows * (uint32_t)sizeof(FastRow), &s.bar);
    }
    if (BITS == 1) {
      const uint32_t total_words = p.n_bits_rows * p.words;
      for (uint32_t i = threadIdx.x; i < total_words; i += blockDim.x) s.bits[i] = __ldg(p.bits + i);
    }
    const uint32_t cbase = blockIdx.x * kEvalCols + threadIdx.x * 4u;   // 4 consecutive columns per lane
    WorkerReg w[kEvalWPT];
    // word = price + b * (0xFFFF - price), two words per 32-bit half of the store.  The odd column's difference is
    // pre-shifted and both prices pre-packed, so a half is two multiply-adds: b1 * (d1 << 16) + (b0 * d0 + (p0 | p1 << 16));
    // b0 * d0 + p0 <= 0xFFFF, so nothing carries into the upper word.  Padding columns are null workers: 0xFFFF.
    uint32_t nd[kEvalWPT];
#pragma unroll
    for (int k = 0; k < kEvalWPT; ++k) {
      const uint32_t col = cbase + k;
      if (col < nw) {
        w[k] = make_worker(__ldg(p.wa + w0 + col), __ldg(p.wb + w0 + col));
        if (p.nacc) w[k].mmask = __ldg(p.nacc + w0 + col);
      } else w[k] = null_worker();
      nd[k] = (0xFFFFu - w[k].price) << ((k & 1) * 16);
    }
    const uint32_t np0 = w[0].price | (w[1].price << 16), np1 = w[2].price | (w[3].price << 16);
    uint2* out = reinterpret_cast<uint2*>(cost + (size_t)r0 * ld + cbase);
    const size_t row_stride = ld / 4;   // in 8-byte units
    const uint32_t sh = p.sign_shift;
    __syncthreads();
    mbar_wait(&s.bar, 0);
    FastRow cur = s.row[0];
    for (uint32_t r = 0; r < nrows; ++r) {
      FastRow nxt = cur;
      if (r + 1 < nrows) nxt = s.row[r + 1];
      uint32_t um[kEvalWPT];
      eval_fast_first<kEvalWPT, BITS>(cur, s.bits, w, p.bits, p.words, um);
      if (cur.n_opts > 1u)
        eval_fast_more<kEvalWPT, BITS>(p.opts_fast + cur.opt_off + 1, cur.n_opts - 1u, s.bits, w, p.bits, p.words, um);
      uint32_t b[kEvalWPT];
#pragma unroll
      for (int k = 0; k < kEvalWPT; ++k)
        b[k] = (um[k] | (w[k].cores - cur.cpu_cores) | (w[k].ram - cur.ram_mb) | (w[k].storage - cur.storage_gb)) >> sh;
      uint2 v;
      v.x = b[1] * nd[1] + (b[0] * nd[0] + np0);
      v.y = b[3] * nd[3] + (b[2] * nd[2] + np1);
      __stcs(out, v);
      out += row_stride;
      cur = nxt;
    }
  } else {
    __shared__ FastStage<ROWS> s;
    const uint32_t r0 = blockIdx.y * ROWS;
    const uint32_t nrows = min(nt - r0, (uint32_t)ROWS);
    if (threadIdx.x == 0) {
      mbar_init(&s.bar, 1);
      mbar_expect_tx(&s.bar, nrows * (uint32_t)sizeof(FastRow));
      bulk_g2s(s.row, p.frows + t0 + r0, nrows * (uint32_t)sizeof(FastRow), &s.bar);
    }
    if (BITS == 1) {
      const uint32_t total_words = p.n_bits_rows * p.words;
      for (uint32_t i = threadIdx.x; i < total_words; i += blockDim.x) s.bits[i] = __ldg(p.bits + i);
    }
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t cbase = blockIdx.x * kEvalCols + (threadIdx.x >> 5) * 128u + lane * 2u;
    WorkerReg w[kEvalWPT];
    uint32_t gw[kEvalWPT], dx[kEvalWPT], dy[kEvalWPT];
  #pragma unroll
    for (int k = 0; k < kEvalWPT; ++k) {
      const uint32_t col = cbase + (k >> 1) * 64u + (k & 1);
      gw[k] = w0 + col;
      if (col < nw) {
        w[k] = make_worker(__ldg(p.wa + w0 + col), __ldg(p.wb + w0 + col));
        if (p.nacc) w[k].mmask = __ldg(p.nacc + w0 + col);
      } else w[k] = null_worker();
      dx[k] = 0xFFFFFFFFu - gw[k];          // infeasible: 0x7FFFFFFF_FFFFFFFF = feasible word + (0/1) * difference
      dy[k] = 0x7FFFFFFFu - w[k].price;
    }
    uint4* out = reinterpret_cast<uint4*>(cost + (size_t)r0 * ld + cbase);
    const size_t row_stride = ld / 2;
    const uint32_t sh = p.sign_shift;
    __syncthreads();            // mbarrier initialised, acceptance words staged
    mbar_wait(&s.bar, 0);
    FastRow cur = s.row[0];
    for (uint32_t r = 0; r < nrows; ++r) {
      FastRow nxt = cur;
      if (r + 1 < nrows) nxt = s.row[r + 1];    // in flight while this row is evaluated
      uint32_t um[kEvalWPT];
      eval_fast_first<kEvalWPT, BITS>(cur, s.bits, w, p.bits, p.words, um);
      if (cur.n_opts > 1u)                      // OR-options (node.rs:420-438): the ask fails only if every option does
        eval_fast_more<kEvalWPT, BITS>(p.opts_fast + cur.opt_off + 1, cur.n_opts - 1u, s.bits, w, p.bits, p.words, um);
      uint4 v0, v1;
      {
        uint32_t o[2 * kEvalWPT];
  #pragma unroll
        for (int k = 0; k < kEvalWPT; ++k) {
          const uint32_t fail = um[k] | (w[k].cores - cur.cpu_cores) | (w[k].ram - cur.ram_mb) | (w[k].storage - cur.storage_gb);
          const uint32_t b = fail >> sh;                                    // 1 when infeasible (sh == 31)
          o[2 * k] = b * dx[k] + gw[k];                                     // feasible: (price << 32) | worker
          o[2 * k + 1] = b * dy[k] + w[k].price;                            // infeasible: 0x7FFFFFFF_FFFFFFFF
        }
        v0 = make_uint4(o[0], o[1], o[2], o[3]);
        v1 = make_uint4(o[4], o[5], o[6], o[7]);
      }
      __stcs(out, v0);
      __stcs(out + 32, v1);     // + 64 columns
      out += row_stride;
      cur = nxt;
    }
  }
}

// The int64 packed cost of a 16-bit tile (pm_build_cost_tile's host output): price << 32 | worker, or
// 0x7FFFFFFF_FFFFFFFF where the word is 0xFFFF.
__global__ void pm_widen_cost(const uint16_t* __restrict__ in, size_t n, size_t ld, uint32_t w0, long long* __restrict__ out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t h = in[i];
    out[i] = h == 0xFFFFu ? kInf : (long long)(((unsigned long long)h << 32) | (w0 + (uint32_t)(i % ld)));
  }
}

// Worker-major acceptance: bit r of nacc[w] is set when pattern row r rejects worker w's model (row 0 never does).
__global__ void pm_worker_nacc(const uint4* __restrict__ wa, const uint32_t* __restrict__ bits, uint32_t words, uint32_t n_rows,
                               uint32_t n, uint32_t* __restrict__ nacc) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4 a = wa[i];
  const uint32_t mid = (a.w & PM_W_HAS_GPU_MODEL) ? a.z : 0u;
  const uint32_t mword = mid / kModelsPerWord, mmask = 1u << (mid % kModelsPerWord);
  uint32_t rej = 0;
  for (uint32_t r = 1; r < n_rows; ++r)
    if (!(__ldg(bits + (size_t)r * words + mword) & mmask)) rej |= 1u << r;
  nacc[i] = rej;
}

// `wp` of every FastRow: the first option's acceptance WORD when rows are one word wide, else its pattern row.
__global__ void pm_bind_rows(FastRow* __restrict__ rows, const DevOptF* __restrict__ opts_fast,
                             const uint32_t* __restrict__ bits, uint32_t words, uint32_t n_asks) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_asks) return;
  const uint32_t prow = opts_fast[rows[t].opt_off].pattern_row;
  rows[t].wp = words == 1u ? bits[prow] : prow;
}

// ------------------------------------------------------------------ argmin
constexpr int kArgThreads = 256;
constexpr int kArgWarps = kArgThreads / 32;
constexpr int kArgRows = 64;                     // rows per CTA

// grid = (ceil(ld / (8*S*64)), ceil(nt / 64)).  All 8 warps of a CTA work on the SAME
// RPW rows at a time, each on its own S*64-column slice (so a CTA touches RPW DRAM
// pages / TLB entries at a time even when rows are megabytes apart); a lane issues
// S*RPW independent 128-bit streaming loads before the first use (8 KB per warp in
// flight at S=8, RPW=2), folds them lane-locally, then one shuffle reduction per
// row.  Per-column "first feasible ask" never leaves the lane's registers; per-row
// (min, count) partials are merged in shared memory and flushed once per CTA.
template <int S, int RPW>
__global__ void __launch_bounds__(kArgThreads)
pm_argmin(const long long* __restrict__ cost, size_t ld, uint32_t nt, uint32_t t0, uint32_t w0,
          uint32_t nw, uint32_t* __restrict__ first_ask, long long* __restrict__ ask_best,
          uint32_t* __restrict__ ask_count) {
  constexpr int kWarpCols = S * 64;
  __shared__ unsigned long long s_best[kArgRows];
  __shared__ uint32_t s_cnt[kArgRows];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t c0 = (blockIdx.x * kArgWarps + warp) * kWarpCols;   // this warp's first column
  const uint32_t r0 = blockIdx.y * kArgRows;
  const uint32_t rows = min((uint32_t)kArgRows, nt - r0);
  for (uint32_t i = threadIdx.x; i < (uint32_t)kArgRows; i += kArgThreads) {
    s_best[i] = (unsigned long long)kInf;
    s_cnt[i] = 0;
  }
  __syncthreads();

  uint32_t cm[S][2];
#pragma unroll
  for (int s = 0; s < S; ++s) cm[s][0] = cm[s][1] = kNone;

  if (c0 < ld) {
    for (uint32_t rr = 0; rr < rows; rr += RPW) {
      longlong2 v[RPW][S];
#pragma unroll
      for (int q = 0; q < RPW; ++q) {
        const uint32_t r = r0 + rr + q;
        const longlong2* rowp = reinterpret_cast<const longlong2*>(cost + (size_t)r * ld);
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const uint32_t col = c0 + s * 64 + lane * 2;
          if (rr + q < rows && col < ld) v[q][s] = __ldcs(rowp + (col >> 1));
          else v[q][s] = make_longlong2(kInf, kInf);
        }
      }
#pragma unroll
      for (int q = 0; q < RPW; ++q) {
        const uint32_t t = t0 + r0 + rr + q;
        long long best = kInf;
        uint32_t cnt = 0;
#pragma unroll
        for (int s = 0; s < S; ++s) {
          best = min(best, min(v[q][s].x, v[q][s].y));
          const bool fx = v[q][s].x != kInf, fy = v[q][s].y != kInf;
          cnt += (uint32_t)fx + (uint32_t)fy;
          cm[s][0] = fx ? min(cm[s][0], t) : cm[s][0];
          cm[s][1] = fy ? min(cm[s][1], t) : cm[s][1];
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          best = min(best, __shfl_xor_sync(0xffffffffu, best, off));
          cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
        }
        if (lane == 0 && cnt) {
          atomicMin(&s_best[rr + q], (unsigned long long)best);
          atomicAdd(&s_cnt[rr + q], cnt);
        }
      }
    }
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const uint32_t col = c0 + s * 64 + lane * 2;
      if (cm[s][0] != kNone && col < nw) atomicMin(first_ask + w0 + col, cm[s][0]);
      if (cm[s][1] != kNone && col + 1 < nw) atomicMin(first_ask + w0 + col + 1, cm[s][1]);
    }
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < rows; i += kArgThreads) {
    if (s_cnt[i]) {
      atomicMin(ask_best + t0 + r0 + i, (long long)s_best[i]);
      atomicAdd(ask_count + t0 + r0 + i, s_cnt[i]);
    }
  }
}

// 16-bit form: one read of a price-word tile (2 B per evaluation), same outputs as pm_argmin.  A lane loads 8 columns per
// 128-bit load, S loads per row (a warp covers S*256 columns, a CTA 8*S*256 <= 65536).  The row minimum is folded on a
// 32-bit key price << 16 | column offset: inside a lane the offset is the compile-time position of the column among the
// lane's own (one IMAD forms the key of the low word, one LOP3 that of the high word), the lane's base offset within the
// CTA's span is added once per row, and the key is widened to the int64 key (price << 32 | worker) only at the per-CTA
// flush.  Infeasible words (0xFFFF) give keys >= 0xFFFF0000 and are neither counted nor folded into first_ask.
template <int S, int RPW>
__global__ void __launch_bounds__(kArgThreads)
pm_argmin16(const uint16_t* __restrict__ cost, size_t ld, uint32_t nt, uint32_t t0, uint32_t w0,
            uint32_t nw, uint32_t* __restrict__ first_ask, long long* __restrict__ ask_best,
            uint32_t* __restrict__ ask_count) {
  constexpr uint32_t kWarpCols = S * 256;
  constexpr uint32_t kCtaCols = kArgWarps * kWarpCols;
  static_assert(kCtaCols <= 65536u, "column offsets are 16 bits");
  constexpr uint32_t kInfeasible = 0xFFFF0000u;   // keys at or above: infeasible words
  __shared__ uint32_t s_best[kArgRows];
  __shared__ uint32_t s_cnt[kArgRows];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t cta_c0 = blockIdx.x * kCtaCols;
  const uint32_t lane_off = warp * kWarpCols + lane * 8u;    // this lane's first column, relative to the CTA's span
  const uint32_t c0 = cta_c0 + lane_off;
  const uint32_t r0 = blockIdx.y * kArgRows;
  const uint32_t rows = min((uint32_t)kArgRows, nt - r0);
  for (uint32_t i = threadIdx.x; i < (uint32_t)kArgRows; i += kArgThreads) {
    s_best[i] = kNone;
    s_cnt[i] = 0;
  }
  __syncthreads();

  uint32_t cm[S][8];
#pragma unroll
  for (int s = 0; s < S; ++s)
#pragma unroll
    for (int j = 0; j < 8; ++j) cm[s][j] = kNone;

  if (cta_c0 + warp * kWarpCols < ld) {
    for (uint32_t rr = 0; rr < rows; rr += RPW) {
      uint4 v[RPW][S];
#pragma unroll
      for (int q = 0; q < RPW; ++q) {
        const uint4* rowp = reinterpret_cast<const uint4*>(cost + (size_t)(r0 + rr + q) * ld);
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const uint32_t col = c0 + s * 256;
          if (rr + q < rows && col < ld) v[q][s] = __ldcs(rowp + (col >> 3));
          else v[q][s] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
        }
      }
#pragma unroll
      for (int q = 0; q < RPW; ++q) {
        const uint32_t t = t0 + r0 + rr + q;
        uint32_t best = kInfeasible, cnt = 0;
#pragma unroll
        for (int s = 0; s < S; ++s) {
          const uint32_t x4[4] = {v[q][s].x, v[q][s].y, v[q][s].z, v[q][s].w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t x = x4[j];
            const uint32_t off = s * 256 + 2 * j;             // lane-relative: s * 256 + 2j (+ 1 for the high word)
            const uint32_t klo = x * 65536u + off;            // (low word << 16) | off
            const uint32_t khi = (x & 0xFFFF0000u) | (off + 1u);
            best = min(best, min(klo, khi));                  // strict order: the lower column wins a tie in price
            const bool flo = klo < kInfeasible, fhi = x < kInfeasible;
            cnt += (uint32_t)flo + (uint32_t)fhi;
            cm[s][2 * j] = flo ? min(cm[s][2 * j], t) : cm[s][2 * j];
            cm[s][2 * j + 1] = fhi ? min(cm[s][2 * j + 1], t) : cm[s][2 * j + 1];
          }
        }
        best += lane_off;                                     // < 0xFFFF0000 + 65536: no carry out of the key
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
          cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        }
        if (lane == 0 && cnt) {
          atomicMin(&s_best[rr + q], best);
          atomicAdd(&s_cnt[rr + q], cnt);
        }
      }
    }
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t col = c0 + s * 256 + j;
        if (cm[s][j] != kNone && col < nw) atomicMin(first_ask + w0 + col, cm[s][j]);
      }
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < rows; i += kArgThreads) {
    if (s_cnt[i]) {   // a counted row has a feasible minimum: key < 0xFFFF0000
      const uint32_t key = s_best[i];
      const unsigned long long wide = ((unsigned long long)(key >> 16) << 32) | (w0 + cta_c0 + (key & 0xFFFFu));
      atomicMin(ask_best + t0 + r0 + i, (long long)wide);
      atomicAdd(ask_count + t0 + r0 + i, s_cnt[i]);
    }
  }
}

// ------------------------------------------------------------------ fused
// Same stripe/row decomposition as pm_build_cost, but the int64 cost never
// leaves the SM: per-row results go through ballots (first-fit cost is the
// worker index, so the row minimum is the lowest set bit), per-worker results
// stay in registers.  Integer-issue-bound, not HBM-bound.
// STATS = false skips the per-ask (min, count) outputs — the reference modes only need the
// per-worker first feasible ask — which removes the ballots from the inner loop.
template <int BITS, bool FAST, bool STATS>
__global__ void __launch_bounds__(kEvalThreads, 2)
pm_fused_eval(EvalParams p, uint32_t t0, uint32_t nt, uint32_t w0, uint32_t nw,
              uint32_t* __restrict__ first_ask, long long* __restrict__ ask_best,
              uint32_t* __restrict__ ask_count) {
  __shared__ EvalStage s;
  __shared__ uint32_t s_cnt[kEvalRows];
  __shared__ uint32_t s_best[kEvalRows];
  const uint32_t r0 = blockIdx.y * kEvalRows;
  const uint32_t r1 = min(nt, r0 + (uint32_t)kEvalRows);
  for (uint32_t i = threadIdx.x; i < (uint32_t)kEvalRows; i += kEvalThreads) {
    s_cnt[i] = 0;
    s_best[i] = kNone;
  }
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t c = blockIdx.x * kEvalCols + threadIdx.x * kEvalWPT;
  WorkerReg w[kEvalWPT];
  load_workers<kEvalWPT>(p, w0, nw, c, w);
  uint32_t first[kEvalWPT];
#pragma unroll
  for (int k = 0; k < kEvalWPT; ++k) first[k] = kNone;
  const uint32_t warp_gw0 = w0 + (c - lane * kEvalWPT);
  for_each_staged_row(s, p, FAST, t0, r0, r1, [&](uint32_t r, const DevAsk& a, uint32_t obegin, bool staged) {
    uint32_t f[kEvalWPT];
    if (FAST && staged) {
      uint32_t fail[kEvalWPT];
      eval_row_fast<kEvalWPT, BITS>(s, a, obegin, w, p.bits, p.words, fail);
#pragma unroll
      for (int k = 0; k < kEvalWPT; ++k) f[k] = ~(uint32_t)((int32_t)fail[k] >> 31);   // all-ones <=> feasible
    } else if (staged) {
      eval_row<kEvalWPT, BITS>(s, a, obegin, w, p.bits, p.words, f);
    } else {
      eval_row_global<kEvalWPT>(p, a, w, f);
    }
    const uint32_t t = t0 + r0 + r;
#pragma unroll
    for (int k = 0; k < kEvalWPT; ++k) first[k] = min(first[k], t | ~f[k]);
    if (STATS) {
      uint32_t cnt = 0, best = kNone;
#pragma unroll
      for (int k = 0; k < kEvalWPT; ++k) {
        const uint32_t b = __ballot_sync(0xffffffffu, f[k] != 0u);
        cnt += (uint32_t)__popc(b);
        if (b) best = min(best, ((uint32_t)__ffs(b) - 1u) * kEvalWPT + k);
      }
      if (cnt && lane == 0) {
        atomicAdd(&s_cnt[r], cnt);
        atomicMin(&s_best[r], warp_gw0 + best);
      }
    }
  });
#pragma unroll
  for (int k = 0; k < kEvalWPT; ++k)
    if (first[k] != kNone) atomicMin(first_ask + w0 + c + k, first[k]);
  if (!STATS) return;
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < r1 - r0; i += kEvalThreads) {
    if (s_cnt[i]) {
      atomicAdd(ask_count + t0 + r0 + i, s_cnt[i]);
      atomicMin(ask_best + t0 + r0 + i, (long long)s_best[i]);
    }
  }
}

// ------------------------------------------------------------------ ask-table conversion
// pm_ask / pm_gpu_opt (ABI form, field-for-field NodeGroupConfiguration + GpuRequirements) ->
// DevAsk / DevOpt / DevOptF, on the device: the upload is a plain memcpy of the caller's tables
// and one pass of these two kernels instead of a host loop.
enum AskStatusBit : uint32_t {
  kAskBadSizes = 1u << 0,   // max_group_size < min_group_size (is_valid, mod.rs:55-60)
  kAskBadRange = 1u << 1,   // opt_off + n_opts out of bounds
  kAskNotSmall = 1u << 2,   // an operand does not fit the fast predicate
  kAskNotSolo = 1u << 3,    // some ask is not min == max == 1
  kAskMaxZero = 1u << 4     // some ask has max_group_size == 0
};

__global__ void pm_ask_counts(const pm_ask* __restrict__ asks, uint32_t n_asks, uint32_t n_opts,
                              uint32_t* __restrict__ counts, uint32_t* __restrict__ status) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_asks) return;
  if (t == n_asks) { counts[t] = 0; return; }
  const pm_ask a = asks[t];
  uint32_t st = 0;
  if (a.max_group_size < a.min_group_size) st |= kAskBadSizes;
  if ((unsigned long long)a.opt_off + a.n_opts > n_opts) st |= kAskBadRange;
  if (!(a.min_group_size == 1 && a.max_group_size == 1)) st |= kAskNotSolo;
  if (a.max_group_size == 0) st |= kAskMaxZero;
  if (st) atomicOr(status, st);
  // every converted ask owns at least one option row: an ask without GPU options gets a neutral one (pm_ask_convert)
  counts[t] = max(((a.flags & PM_A_HAS_REQ) && !(st & kAskBadRange)) ? a.n_opts : 0u, 1u);
}

__global__ void pm_ask_convert(const pm_ask* __restrict__ asks, const pm_gpu_opt* __restrict__ opts,
                               uint32_t n_asks, const uint32_t* __restrict__ new_off,
                               DevAsk* __restrict__ dasks, DevOpt* __restrict__ dopts,
                               DevOptF* __restrict__ doptsf, uint32_t* __restrict__ amin,
                               uint32_t* __restrict__ amax, uint32_t* __restrict__ status,
                               uint32_t* __restrict__ max_row, FastRow* __restrict__ frows) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_asks) return;
  const pm_ask a = asks[t];
  DevAsk d;
  d.n_opts = 0; d.cpu_cores = 0; d.ram_mb = 0; d.storage_gb = 0; d.pad0 = 0; d.pad1 = 0;
  const bool has_req = (a.flags & PM_A_HAS_REQ) != 0;
  uint32_t need = kCandBit;
  const uint32_t n_rows = new_off[t + 1] - new_off[t];                  // >= 1
  // option rows that come from the caller (none are read when pm_ask_counts found a range out of bounds: the call fails)
  const bool bad_range = (*reinterpret_cast<volatile uint32_t*>(status) & kAskBadRange) != 0u;
  const uint32_t n_eff = (has_req && !bad_range) ? min(a.n_opts, n_rows) : 0u;
  if (has_req) {
    need |= PM_W_HAS_SPECS;
    if (a.flags & PM_A_REQ_CPU) need |= PM_W_HAS_CPU;
    if ((a.flags & PM_A_REQ_CPU) && (a.flags & PM_A_REQ_CPU_CORES)) { need |= PM_W_HAS_CPU_CORES; d.cpu_cores = a.cpu_cores; }
    if (a.flags & PM_A_REQ_RAM) { need |= PM_W_HAS_RAM; d.ram_mb = a.ram_mb; }
    if (a.flags & PM_A_REQ_STORAGE) { need |= PM_W_HAS_STORAGE; d.storage_gb = a.storage_gb; }
    if (a.n_opts) need |= PM_W_HAS_GPU;
  }
  d.n_opts = n_rows;
  if (a.max_group_size == 0) need |= kNeverBit;   // first-fit with max_group_size == 0 takes nobody (mod.rs:555-556)
  d.need = need;
  d.opt_off = new_off[t];
  uint32_t st = 0, mrow = 0;
  if ((d.cpu_cores | d.ram_mb | d.storage_gb) >= kSign) st |= kAskNotSmall;
  for (uint32_t o = 0; o < n_eff; ++o) {
    const pm_gpu_opt q = opts[a.opt_off + o];
    DevOpt x;
    x.need = 0;
    x.count_mask = (q.present & PM_O_COUNT) ? 0xFFFFFFFFu : 0u;
    x.count = (q.present & PM_O_COUNT) ? q.count : 0u;
    uint32_t mem_lo = 0, mem_hi = 0xFFFFFFFFu, tot_lo = 0, tot_hi = 0xFFFFFFFFu;
    if (q.present & PM_O_MEM) mem_lo = max(mem_lo, q.memory_mb);
    if (q.present & PM_O_MEM_MIN) mem_lo = max(mem_lo, q.memory_mb_min);
    if (q.present & PM_O_MEM_MAX) mem_hi = q.memory_mb_max;
    if (q.present & (PM_O_MEM | PM_O_MEM_MIN | PM_O_MEM_MAX)) x.need |= PM_W_HAS_GPU_MEM;
    if (q.present & PM_O_TOT_MIN) tot_lo = q.total_memory_min;
    if (q.present & PM_O_TOT_MAX) tot_hi = q.total_memory_max;
    if (mem_lo > mem_hi) { x.need |= kNeverBit; mem_lo = 0; mem_hi = 0xFFFFFFFFu; }
    if (tot_lo > tot_hi) { x.need |= kTotInvalidBit; tot_lo = 0; tot_hi = 0xFFFFFFFFu; }
    x.mem_lo = mem_lo; x.mem_span = mem_hi - mem_lo;
    x.tot_lo = tot_lo; x.tot_span = tot_hi - tot_lo;
    x.pattern_row = 0;
    if (q.present & PM_O_MODEL) {
      x.need |= PM_W_HAS_GPU_MODEL;
      x.pattern_row = q.pattern_id + 1;
      mrow = max(mrow, x.pattern_row);
    }
    dopts[d.opt_off + o] = x;
    DevOptF f;
    const uint32_t need_all = need | x.need;
    f.m = key_bits(need_all); f.v = f.m;
    if (q.present & PM_O_COUNT) {
      if (q.count >= 65536u) st |= kAskNotSmall;
      f.m |= 0xFFFFu << kKeyCountShift;
      f.v |= (q.count & 0xFFFFu) << kKeyCountShift;
    }
    if (mem_lo >= kSign || tot_lo >= kSign) st |= kAskNotSmall;
    f.mem_lo = mem_lo; f.mem_hi = min(mem_hi, 0x7FFFFFFFu);
    f.tot_lo = tot_lo; f.tot_hi = min(tot_hi, 0x7FFFFFFFu);
    f.pattern_row = x.pattern_row; f.pad = 0;
    doptsf[d.opt_off + o] = f;
  }
  if (n_eff == 0u) {
    // no GPU clause (requirements.gpu empty, or no requirements at all): one neutral option row — it accepts every
    // worker, so the ask's presence bits and scalar thresholds decide alone — keeps the evaluation loops free of an
    // option-less special case
    DevOpt x;
    x.need = 0; x.count_mask = 0; x.count = 0; x.mem_lo = 0; x.mem_span = 0xFFFFFFFFu; x.tot_lo = 0; x.tot_span = 0xFFFFFFFFu;
    x.pattern_row = 0;
    dopts[d.opt_off] = x;
    DevOptF f;
    f.m = key_bits(need); f.v = f.m;
    f.mem_lo = 0; f.mem_hi = 0x7FFFFFFFu; f.tot_lo = 0; f.tot_hi = 0x7FFFFFFFu; f.pattern_row = 0; f.pad = 0;
    doptsf[d.opt_off] = f;
  }
  dasks[t] = d;
  {
    const DevOptF f = doptsf[d.opt_off];   // written above by this thread
    FastRow fr;
    fr.m = f.m; fr.v = f.v; fr.mem_lo = f.mem_lo; fr.mem_hi = f.mem_hi;
    fr.tot_lo = f.tot_lo; fr.tot_hi = f.tot_hi; fr.wp = f.pattern_row; fr.n_opts = n_rows;
    fr.cpu_cores = d.cpu_cores; fr.ram_mb = d.ram_mb; fr.storage_gb = d.storage_gb; fr.opt_off = d.opt_off;
    frows[t] = fr;
  }
  amin[t] = a.min_group_size;
  amax[t] = a.max_group_size;
  if (st) atomicOr(status, st);
  if (mrow) atomicMax(max_row, mrow);
}

// ------------------------------------------------------------------ small utilities
__global__ void pm_fill_u32(uint32_t* p, uint32_t v, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void pm_fill_i64(long long* p, long long v, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void pm_iota_u32(uint32_t* p, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = (uint32_t)i;
}
__global__ void pm_scatter_flags(uint4* wa, const uint32_t* idx, const uint32_t* flags, uint32_t n, uint32_t n_workers) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && idx[i] < n_workers) wa[idx[i]].w = flags[i];
}

// pm_update_workers: rows that changed since the last pass, scattered into the resident table
__global__ void pm_scatter_rows(uint4* wa, uint4* wb, double* lat, double* lon, const uint32_t* __restrict__ idx,
                                const uint4* __restrict__ a, const uint4* __restrict__ b, const double* __restrict__ la,
                                const double* __restrict__ lo, uint32_t n, uint32_t n_workers) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t w = idx[i];
  if (w >= n_workers) return;
  wa[w] = a[i];
  wb[w] = b[i];
  if (lat) { lat[w] = la[i]; lon[w] = lo[i]; }
}

// Do all workers satisfy the fast-path operand limits (values < 2^31, gpu count < 2^16,
// count * memory_mb < 2^31 without wrapping)?  Clears *ok otherwise.  Clears *narrow when a
// worker's ext_ask_price does not fit a 16-bit cost word (> 0xFFFE: 0xFFFF means infeasible).
__global__ void pm_check_worker_ranges(const uint4* __restrict__ wa, const uint4* __restrict__ wb,
                                       uint32_t n, uint32_t* __restrict__ ok, uint32_t* __restrict__ narrow) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4 a = wa[i], b = wb[i];
  bool small = (b.x | b.y | b.z) < kSign;
  if (a.w & PM_W_HAS_GPU_COUNT) small &= a.x < 65536u;
  if (a.w & PM_W_HAS_GPU_MEM) small &= a.y < kSign;
  if ((a.w & PM_W_HAS_GPU_COUNT) && (a.w & PM_W_HAS_GPU_MEM))
    small &= (unsigned long long)a.x * (unsigned long long)a.y < (unsigned long long)kSign;
  if (!small) *ok = 0u;
  if (b.w > 0xFFFEu) *narrow = 0u;
}

// ------------------------------------------------------------------ resolution
// Sort key of a worker: its (first feasible) ask; in proximity mode with solo
// groups the key also orders located workers first (seed rule, mod.rs:526-530).
__global__ void pm_make_keys(const uint32_t* __restrict__ cur, const uint4* __restrict__ wa,
                             uint32_t n_workers, uint32_t shift, uint32_t* __restrict__ keys,
                             uint32_t* __restrict__ hist) {
  uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_workers) return;
  uint32_t c = cur[w], k = kNone;
  if (c != kNone) {
    k = c << shift;
    if (shift) k |= (wa[w].w & PM_W_HAS_LOC) ? 0u : 1u;
    atomicAdd(hist + k, 1u);
  }
  keys[w] = k;
}

// any configuration whose member count leaves an under-filled tail
// (0 < K mod max < min: the tail group is not formed, mod.rs:517,564)?
__global__ void pm_check_tails(const uint32_t* __restrict__ hist, const uint32_t* __restrict__ amin,
                               const uint32_t* __restrict__ amax, uint32_t n_asks,
                               uint32_t* __restrict__ any_bad) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_asks) return;
  const uint32_t mx = amax[c];
  if (mx == 0) return;
  const uint32_t r = hist[c] % mx;
  if (r != 0 && r < amin[c]) *any_bad = 1u;
}

struct SweepParams {
  EvalParams ev;
  uint32_t* cur;             // [W] current ask of each worker
  uint32_t* base_len;        // [T] members still in the sorted base segment
  const uint32_t* seg_start; // [T]
  const uint32_t* order;     // [W] workers sorted by (ask, index)
  uint32_t* xhead;           // [T] list of workers bumped into the ask
  uint32_t* xnext;           // [W]
  uint32_t* xcount;          // [T]
  const uint32_t* amin;
  const uint32_t* amax;
  uint32_t* popped;          // [W] scratch
  uint32_t* n_bumped;
  const uint32_t* any_bad;   // written by pm_check_tails: 0 = no configuration has an under-filled tail, nothing to do
};

// Sequential-in-priority sweep (single CTA): configurations are final in
// increasing priority index; the first one with an under-filled tail hands its
// last `K mod max` members (largest canonical index — groups are cut from the
// front, mod.rs:554-561) to their next feasible configuration.
__global__ void __launch_bounds__(1024) pm_sweep(SweepParams p) {
  __shared__ uint32_t s_first_bad, s_npop;
  if (*p.any_bad == 0u) return;   // the common case costs one launch, not a host round trip
  const uint32_t T = p.ev.n_asks;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  uint32_t c_lo = 0;
  while (c_lo < T) {
    if (tid == 0) s_first_bad = kNone;
    __syncthreads();
    const uint32_t c = c_lo + tid;
    if (c < T) {
      const uint32_t mx = p.amax[c];
      if (mx) {
        const uint32_t r = (p.base_len[c] + p.xcount[c]) % mx;
        if (r && r < p.amin[c]) atomicMin(&s_first_bad, c);
      }
    }
    __syncthreads();
    const uint32_t cb = s_first_bad;
    if (cb == kNone) {
      c_lo += 1024;
      continue;
    }
    if (tid == 0) {
      uint32_t bl = p.base_len[cb], xc = p.xcount[cb];
      const uint32_t r = (bl + xc) % p.amax[cb];
      for (uint32_t i = 0; i < r; ++i) {
        uint32_t bx = kNone, bprev = kNone, prev = kNone;  // largest index among bumped-in
        for (uint32_t x = p.xhead[cb]; x != kNone; prev = x, x = p.xnext[x])
          if (bx == kNone || x > bx) { bx = x; bprev = prev; }
        const uint32_t bw = bl ? p.order[p.seg_start[cb] + bl - 1] : kNone;
        uint32_t take;
        if (bx != kNone && (bw == kNone || bx > bw)) {
          take = bx;
          if (bprev == kNone) p.xhead[cb] = p.xnext[bx];
          else p.xnext[bprev] = p.xnext[bx];
          --xc;
        } else {
          take = bw;
          --bl;
        }
        p.popped[i] = take;
      }
      p.base_len[cb] = bl;
      p.xcount[cb] = xc;
      s_npop = r;
    }
    __syncthreads();
    const uint32_t npop = s_npop;
    for (uint32_t i = warp; i < npop; i += 32) {
      const uint32_t w = p.popped[i];
      const WorkerReg wr = make_worker(p.ev.wa[w], p.ev.wb[w]);
      uint32_t found = kNone;
      for (uint32_t cbase = cb + 1; cbase < T; cbase += 32) {
        const uint32_t c2 = cbase + lane;
        bool ok = false;
        if (c2 < T) ok = ask_meets(p.ev.asks[c2], p.ev.opts, wr, p.ev.bits, p.ev.words);
        const uint32_t b = __ballot_sync(0xffffffffu, ok);
        if (b) {
          found = cbase + (uint32_t)__ffs(b) - 1u;
          break;
        }
      }
      if (lane == 0) {
        p.cur[w] = found;
        if (found != kNone) {
          const uint32_t old = atomicExch(&p.xhead[found], w);
          p.xnext[w] = old;
          atomicAdd(&p.xcount[found], 1u);
        }
        atomicAdd(p.n_bumped, 1u);
      }
    }
    __syncthreads();
    c_lo = cb + 1;
  }
}

// groups per bin (bin = ask << shift | located-first bit): full chunks of `max`
// plus the tail when it reaches `min` (mod.rs:545-566), plus the empty group a
// min_group_size == 0 configuration produces on its last iteration (:564,:606).
__global__ void pm_count_groups(const uint32_t* __restrict__ hist, const uint32_t* __restrict__ amin,
                                const uint32_t* __restrict__ amax, uint32_t n_bins, uint32_t shift,
                                uint32_t* __restrict__ ngroups) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_bins) return;
  const uint32_t c = b >> shift, mx = amax[c], mn = amin[c], K = hist[b];
  uint32_t g = 0;
  if (mx) {
    g = K / mx;
    const uint32_t r = K % mx;
    if (r && r >= mn) ++g;
  }
  if (mn == 0 && (!shift || (b & 1u))) ++g;
  ngroups[b] = g;
}

// one thread per sorted position: worker -> (group, ask); group heads write the
// group table.  Positions past the formed groups of a bin (an unformed tail can
// only exist if the sweep was skipped by the caller) stay unassigned.
__global__ void pm_emit_workers(const uint32_t* __restrict__ keys_sorted,
                                const uint32_t* __restrict__ order, const uint32_t* __restrict__ n_assigned_dev,
                                const uint32_t* __restrict__ hist,
                                const uint32_t* __restrict__ seg_start,
                                const uint32_t* __restrict__ group_base,
                                const uint32_t* __restrict__ amin, const uint32_t* __restrict__ amax,
                                uint32_t shift, uint32_t* __restrict__ worker_group,
                                uint32_t* __restrict__ worker_ask, uint32_t* __restrict__ group_ask,
                                uint32_t* __restrict__ group_off) {
  uint32_t pidx = blockIdx.x * blockDim.x + threadIdx.x;
  if (pidx >= *n_assigned_dev) return;   // launched over all workers: no host read of the count
  const uint32_t b = keys_sorted[pidx], c = b >> shift, w = order[pidx];
  const uint32_t mx = amax[c], K = hist[b], r = pidx - seg_start[b];
  if (mx == 0) return;
  const uint32_t full = K / mx, rem = K % mx;
  if (r >= full * mx && rem < amin[c]) return;  // unformed tail
  const uint32_t g = group_base[b] + r / mx;
  worker_group[w] = g;
  worker_ask[w] = c;
  if (r % mx == 0) {
    group_ask[g] = c;
    group_off[g] = pidx;
  }
}

// the trailing empty group of min_group_size == 0 configurations
__global__ void pm_emit_empty_groups(const uint32_t* __restrict__ hist,
                                     const uint32_t* __restrict__ seg_start,
                                     const uint32_t* __restrict__ group_base,
                                     const uint32_t* __restrict__ ngroups,
                                     const uint32_t* __restrict__ amin, uint32_t n_bins,
                                     uint32_t shift, uint32_t* __restrict__ group_ask,
                                     uint32_t* __restrict__ group_off) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_bins) return;
  const uint32_t c = b >> shift;
  if (amin[c] != 0 || (shift && !(b & 1u))) return;
  const uint32_t g = group_base[b] + ngroups[b] - 1;
  group_ask[g] = c;
  group_off[g] = seg_start[b] + hist[b];
}

// members of a group in BTreeSet<String> order (mod.rs:63-69): position = number
// of members whose address rank is smaller.
__global__ void pm_order_members(const uint32_t* __restrict__ order, const uint32_t* __restrict__ n_assigned_dev,
                                 const uint32_t* __restrict__ worker_group,
                                 const uint32_t* __restrict__ group_off,
                                 const uint32_t* __restrict__ addr_rank,
                                 uint32_t* __restrict__ members) {
  uint32_t pidx = blockIdx.x * blockDim.x + threadIdx.x;
  if (pidx >= *n_assigned_dev) return;
  const uint32_t w = order[pidx];
  const uint32_t g = worker_group[w];
  if (g == kNone) { members[pidx] = w; return; }
  const uint32_t gs = group_off[g], ge = group_off[g + 1];
  uint32_t pos = 0;
  // without address ranks the row index stands in for the address order
  const uint32_t mine = addr_rank ? addr_rank[w] : w;
  for (uint32_t q = gs; q < ge; ++q) {
    const uint32_t o = order[q];
    pos += ((addr_rank ? addr_rank[o] : o) < mine) ? 1u : 0u;
  }
  members[gs + pos] = w;
}

// The CSR end marker group_off[G] and the pass's scalars {G, members, bumped}, written on the device so the
// resolution chain needs no host round trip before its last kernel.
__global__ void pm_close_groups(const uint32_t* __restrict__ n_groups_dev, const uint32_t* __restrict__ n_assigned_dev,
                                const uint32_t* __restrict__ n_bumped_dev, uint32_t* __restrict__ group_off,
                                uint32_t* __restrict__ scalars) {
  const uint32_t G = *n_groups_dev, M = *n_assigned_dev;
  group_off[G] = M;
  scalars[0] = G;
  scalars[1] = M;
  scalars[2] = *n_bumped_dev;
}

// ------------------------------------------------------------------ multi-GPU exchange (SURVEY 8e)
// One rank's contribution to the single collective of a sharded pass, packed into one buffer:
//   [ ask_best int64[T] | ask_count u32[T] | first_ask of the rank's own worker range u32[per] ]
// (`per` = ceil(W / ranks): every rank sends the same size; the last rank's tail is padding.)
__global__ void pm_xchg_pack(const uint32_t* __restrict__ first_ask_shard, uint32_t nw, uint32_t per,
                             const long long* __restrict__ ask_best, const uint32_t* __restrict__ ask_count, uint32_t T,
                             unsigned char* __restrict__ send) {
  long long* s_best = reinterpret_cast<long long*>(send);
  uint32_t* s_cnt = reinterpret_cast<uint32_t*>(send + (size_t)T * 8);
  uint32_t* s_first = s_cnt + T;
  const size_t n = (size_t)max(T, per);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    if (i < T) { s_best[i] = ask_best[i]; s_cnt[i] = ask_count[i]; }
    if (i < per) s_first[i] = i < nw ? first_ask_shard[i] : kNone;
  }
}

// After the all-gather: every rank folds the `ranks` contributions into the same global arrays — per ask the
// packed (cost, worker) minimum and the feasible-count sum, per worker the first feasible ask from its owner.
__global__ void pm_xchg_unpack(const unsigned char* __restrict__ recv, uint32_t ranks, size_t stride, uint32_t per,
                               uint32_t W, uint32_t T, uint32_t* __restrict__ first_ask,
                               long long* __restrict__ ask_best, uint32_t* __restrict__ ask_count) {
  const size_t n = (size_t)max(T, W);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    if (i < T) {
      long long best = kInf;
      uint32_t cnt = 0;
      for (uint32_t r = 0; r < ranks; ++r) {
        const unsigned char* base = recv + (size_t)r * stride;
        best = min(best, reinterpret_cast<const long long*>(base)[i]);
        cnt += reinterpret_cast<const uint32_t*>(base + (size_t)T * 8)[i];
      }
      ask_best[i] = best;
      ask_count[i] = cnt;
    }
    if (i < W) {
      const uint32_t r = (uint32_t)(i / per);
      const uint32_t* f = reinterpret_cast<const uint32_t*>(recv + (size_t)r * stride + (size_t)T * 12);
      first_ask[i] = f[i - (size_t)r * per];
    }
  }
}

}  // namespace pm
