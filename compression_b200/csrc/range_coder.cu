// Range coder for sm_100a: one CTA per code stream, the serial recurrence alone on one warp.
//
// Replaces (paths relative to /root/reference/tensorflow_compression):
//   cc/lib/range_coder.cc:37-307, cc/lib/range_coder.h:79-282          the coder
//   cc/kernels/range_coder_kernels.cc:110-164,168-322,334-471           multi-stream ops
//   cc/kernels/range_coding_kernels.cc:60-379 (+ _util.cc:34-91)        legacy single-stream ops
//
// ENCODER.  The reference emits bytes through a delayed-carry state machine.  Its output is exactly the
// big-number sum  SUM_k a_k * 2^-(16 r_k + 32)  of the per-symbol interval offsets a_k (r_k = number of 16-bit
// renormalisations before symbol k) followed by a short flush; only the recurrence on the interval size is
// inherently serial.  Per stream (encode_kernel, six warps):
//   * gather warps: coalesced symbol loads three passes ahead, fused quantisation, range checks, escape expansion
//     (an escaping symbol is followed by the records of its Elias-gamma bits), table gathers, operand pre-scaling;
//   * chain warp: nothing but the recurrence on the UN-renormalised span (EncChain::step: IADD3 -> IMAD.WIDE ->
//     funnel shift -> IADD3, no select between the multiplies), one entry {L, s'} per Encode;
//   * drain warp: base, carries, emitted 16-bit words and word count are prefix computations over those entries
//     (EncDrain: a warp scan over the maps x -> (x << S) + A), written as unresolved words + one carry bit each;
//   * finalize: warp-wide carry-lookahead over 32-word groups, RangeEncoder::Finalize's tail rule, compaction.
// DECODER.  Same recurrence plus a CDF search per symbol (decode_kernel, three warps: prepare / chain / resolve):
// pre-scaled search keys, a 64-key window per row around its median evaluated two keys per lane with one IMAD.HI
// each and two warp reductions; the symbol index itself is recovered off the chain by the resolve warp.
// The one-warp-per-stream helpers further down (ByteWindow, dec_symbol) serve the legacy single-stream ops only.
#include <algorithm>
#include <cstring>
#include <vector>

#include <cstring>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace tfcb {
namespace {

constexpr unsigned kFull = 0xFFFFFFFFu;

// ---------------------------------------------------------------------------------------------
// Lookup tables
// ---------------------------------------------------------------------------------------------
struct HostRow {
  int32_t start;  // index of cdf[0] inside the lookup buffer
  int32_t ncdf;   // number of cdf entries (bins + 1)
  int32_t prec;   // signed precision entry
};

// meta = ncdf | |precision| << 24 | overflow << 31
__host__ __device__ inline int row_ncdf(int meta) { return meta & 0xFFFFFF; }
__host__ __device__ inline int row_prec(int meta) { return (meta >> 24) & 0x1F; }
__host__ __device__ inline bool row_ovf(int meta) { return meta < 0; }

// Grammar of range_coder_kernels.cc:110-137 (one row) and :139-164 (1-D / 2-D containers).
int scan_row(const int32_t* base, const int32_t* end, const int32_t** cur, std::vector<HostRow>* rows) {
  const int32_t* p = *cur;
  if (end - p < 3) return fail(TFCB_INVALID_ARGUMENT, "CDF ended prematurely.");
  const int64_t ap = p[0] < 0 ? -(int64_t)p[0] : (int64_t)p[0];
  if (ap < 1 || ap >= 17)
    return fail(TFCB_INVALID_ARGUMENT, "precision=%lld not in range [1, 17)", (long long)ap);
  const int32_t last = 1 << ap;
  const int32_t* first = p;
  if (p[1] != 0) return fail(TFCB_INVALID_ARGUMENT, "CDF must start with 0.");
  p += 1;
  for (;;) {
    ++p;
    if (p == end) return fail(TFCB_INVALID_ARGUMENT, "CDF must end with 1 << precision.");
    if (p[0] < p[-1]) return fail(TFCB_INVALID_ARGUMENT, "CDF must be monotonically increasing.");
    if (*p == last) break;
  }
  ++p;
  rows->push_back(HostRow{(int32_t)(first + 1 - base), (int32_t)(p - first - 1), first[0]});
  while (p != end && *p == last) ++p;
  *cur = p;
  return TFCB_OK;
}

int parse_lookup(const int32_t* lookup, int64_t len, int64_t cols, std::vector<HostRow>* rows) {
  rows->clear();
  if (len < 0 || (len > 0 && lookup == nullptr))
    return fail(TFCB_INVALID_ARGUMENT, "`lookup` is null");
  if (len >= (1ll << 31)) return fail(TFCB_INVALID_ARGUMENT, "`lookup` too large");
  if (cols < 0 || (cols > 0 && len % cols != 0))
    return fail(TFCB_INVALID_ARGUMENT, "`lookup` must be rank 1 or 2");
  const int32_t* end = lookup + len;
  for (const int32_t* cur = lookup; cur != end;) {
    const int32_t* row_end = cols > 0 ? cur + cols : end;
    TFCB_TRY(scan_row(lookup, row_end, &cur, rows));
    if (cols > 0 && cur != row_end)
      return fail(TFCB_INVALID_ARGUMENT, "CDF must end with 1 << precision.");
  }
  return TFCB_OK;
}

struct DeviceLookup {
  int32_t* lookup = nullptr;  // device copy of the raw table
  int2* rows = nullptr;       // {start, meta}
  uint2* pairs = nullptr;     // decoder: per cdf entry {c', addend_hi} so that hi32(span*c' + {c',addend_hi}) = T(c) - 1
  int4* rows4 = nullptr;      // decoder: {key segment start, meta, first window index, irregular}
  long long n_pairs = 0;
  int zero_win = 0;  // key index of the all-zero window (decoder tables only)
  int n_rows = 0;
  long long len = 0;
  bool any_overflow = false;
  int max_prec = 0;
  int uniform_prec = 0;  // > 0 when every row shares one precision

  int upload(const int32_t* lookup_host, int64_t len_, int64_t cols, cudaStream_t s, bool for_decoder = false) {
    const int64_t len = len_;
    std::vector<HostRow> hr;
    TFCB_TRY(parse_lookup(lookup_host, len, cols, &hr));
    n_rows = (int)hr.size();
    this->len = len_;
    std::vector<int2> meta(std::max<size_t>(hr.size(), 1));
    for (size_t i = 0; i < hr.size(); ++i) {
      const int ap = hr[i].prec < 0 ? -hr[i].prec : hr[i].prec;
      any_overflow |= hr[i].prec < 0;
      max_prec = std::max(max_prec, ap);
      uniform_prec = (i == 0 || uniform_prec == ap) ? ap : -1;
      meta[i].x = hr[i].start;
      meta[i].y = hr[i].ncdf | (ap << 24) | (hr[i].prec < 0 ? (int)0x80000000 : 0);
    }
    if (uniform_prec < 0) uniform_prec = 0;
    TFCB_TRY(dev_alloc((void**)&lookup, std::max<int64_t>(len, 1) * sizeof(int32_t), s));
    TFCB_TRY(dev_alloc((void**)&rows, meta.size() * sizeof(int2), s));
    if (len > 0)
      TFCB_CUDA_TRY(cudaMemcpyAsync(lookup, lookup_host, len * sizeof(int32_t),
                                    cudaMemcpyHostToDevice, s));
    TFCB_CUDA_TRY(cudaMemcpyAsync(rows, meta.data(), meta.size() * sizeof(int2),
                                  cudaMemcpyHostToDevice, s));
    std::vector<uint2> hp;
    std::vector<int4> hr4;
    if (for_decoder) {
      // Pre-scaled search keys: B'(c) = floor(size*c/2^p) - 1 = hi32(span*c' + {c', 0xFFFFFFFF}) with
      // c' = c << (32-p); c == 2^p -> {0xFFFFFFFF, 0} (B' = span = size - 1).  Every row gets its own padded
      // segment: keys of cdf[0..n], then "full" keys up to index 64, so that the 64-key search window
      // [wfirst, wfirst + 63] (centred on the row's median, wfirst >= 1) never needs clamping.
      // Rows with zero-width bins at either end are marked irregular: slow path only.
      hr4.resize(meta.size());
      for (size_t i = 0; i < hr.size(); ++i) {
        const int ap = hr[i].prec < 0 ? -hr[i].prec : hr[i].prec;
        const int n = hr[i].ncdf - 1;
        const int pstart = (int)hp.size();
        int median = n, irregular = 0;
        for (int e = 0; e <= n; ++e) {
          const uint32_t c = (uint32_t)lookup_host[hr[i].start + e];
          hp.push_back((c == (1u << ap)) ? make_uint2(0xFFFFFFFFu, 0u) : make_uint2(c << (32 - ap), 0xFFFFFFFFu));
          if (e >= 1 && c == 0u) irregular = 1;
          if (e >= 1 && e < n && c == (1u << ap)) irregular = 1;  // trailing zero-width bins
          if (e >= 1 && median == n && c >= (1u << ap) / 2) median = e;
        }
        for (int e = n + 1; e <= 64; ++e) hp.push_back(make_uint2(0xFFFFFFFFu, 0u));
        int wfirst = median - 31;
        if (wfirst > n - 63) wfirst = n - 63;
        if (wfirst < 1) wfirst = 1;
        hr4[i] = make_int4(pstart, meta[i].y, wfirst, irregular);
      }
      // window of keys whose bound is 0: used for irregular rows so that the chain always takes the slow path
      zero_win = (int)hp.size();
      for (int e = 0; e < 64; ++e) hp.push_back(make_uint2(0u, 0u));
      n_pairs = (long long)hp.size();
      TFCB_TRY(dev_alloc((void**)&pairs, hp.size() * sizeof(uint2), s));
      TFCB_TRY(dev_alloc((void**)&rows4, hr4.size() * sizeof(int4), s));
      TFCB_CUDA_TRY(cudaMemcpyAsync(pairs, hp.data(), hp.size() * sizeof(uint2), cudaMemcpyHostToDevice, s));
      TFCB_CUDA_TRY(cudaMemcpyAsync(rows4, hr4.data(), hr4.size() * sizeof(int4), cudaMemcpyHostToDevice, s));
    }
    // the host vectors die at return: make sure the copies have been staged
    TFCB_CUDA_TRY(cudaStreamSynchronize(s));
    return TFCB_OK;
  }
  void release(cudaStream_t s) {
    dev_free(lookup, s);
    dev_free(rows, s);
    dev_free(pairs, s);
    dev_free(rows4, s);
    lookup = nullptr;
    rows = nullptr;
    pairs = nullptr;
    rows4 = nullptr;
  }
};

// ---------------------------------------------------------------------------------------------
// Encoder state and serial recurrence
// ---------------------------------------------------------------------------------------------
// Per stream the arena holds the UNRESOLVED 16-bit words (`words`) and one carry bit per word
// (`cbits`, bit w = "a carry left the 32-bit window while word w was its top half", i.e. +1 into
// word w-1; bit `cnt` is the pending carry of the not yet emitted top word).
struct EncState {
  uint32_t base;  // low end of the interval (32-bit window, wraps), renormalised
  uint32_t span;  // size - 1, renormalised (what RangeEncoder::Finalize looks at)
  uint32_t cnt;   // 16-bit words appended so far (a stream holds < 2^31 words = 4 GB)
  uint32_t raw;   // size - 1 BEFORE the renormalisation that followed the last symbol (what the chain resumes from)
};

// THE RECURRENCE.  The reference keeps (base, size - 1) and, after every Encode, multiplies both by 2^16 when
// size - 1 < 2^16 (range_coder.cc:69-84).  Only the interval SIZE feeds back into the next symbol, and the
// renormalisation is a select between two multiplies on that dependent chain.  Here the chain carries the
// UN-renormalised span `s` of the last symbol and never materialises the shifted one:
//
//   r    = s < 2^16                                 (the renormalisation the reference did after the last symbol)
//   Q(c) = s * ch + ch,   ch = c << (16 - p)        (64-bit: (s + 1) * c * 2^(16-p); c = 2^p fits: ch = 2^16)
//   floor(size * c / 2^p) = r ? Q : Q >> 16         (size = (s + 1) << 16r; exact; low 32 bits)
//   L = that for `lower`, U = that for `upper`;   s' = U - L - 1   (mod 2^32: a full-range symbol at size 2^32 wraps
//                                                                   to the right value)
// i.e. per symbol the dependent chain is  IADD3 -> IMAD.WIDE -> SHF (funnel by 0 or 16) -> IADD3, with the predicate
// of the shift amount evaluated beside the multiply -- no select between two multiplies.  {L, s'} per Encode is
// all the chain produces; the interval's low end, the carries, the emitted words and the word count are PREFIX
// computations over those entries and are done by the drain warp, 32 entries at a time (EncDrain).
// (Formula checked against the reference's on random triples: precisions 1..16, full-range, single-count and
// top-hugging symbols, from the initial state; the GPU tests compare whole streams with the compiled reference.)

// Pre-scaled operands of one Encode(lower, upper, p): {lower << (16-p), 0, upper << (16-p), 0}.  The zeros are
// the high halves of the two multiply-adds' 64-bit addends: one 128-bit shared-memory load puts each bound's
// addend in a register pair of its own.
__device__ __forceinline__ uint4 enc_operands(uint32_t lower, uint32_t upper, uint32_t p) {
  const uint32_t sh = 16u - p;
  return make_uint4(lower << sh, 0u, upper << sh, 0u);
}

struct EncChain {
  uint32_t s;  // un-renormalised span after the last symbol

  // One Encode(lower, upper, precision) of range_coder.cc:37-264 -> the entry {L, s'}.
  __device__ __forceinline__ uint2 step(uint2 ol, uint2 oh) {
    const unsigned long long ql = (unsigned long long)s * ol.x + (((unsigned long long)ol.y << 32) | ol.x);
    const unsigned long long qu = (unsigned long long)s * oh.x + (((unsigned long long)oh.y << 32) | oh.x);
    const uint32_t shift = (s < 65536u) ? 0u : 16u;
    const uint32_t L = __funnelshift_r((uint32_t)ql, (uint32_t)(ql >> 32), shift);
    const uint32_t U = __funnelshift_r((uint32_t)qu, (uint32_t)(qu >> 32), shift);
    s = U - L - 1u;
    return make_uint2(L, s);
  }
  __device__ __forceinline__ uint2 step(uint4 o) { return step(make_uint2(o.x, o.y), make_uint2(o.z, o.w)); }
};

// x << s for s in [0, 32] (s == 32 gives 0): one funnel shift.
__device__ __forceinline__ uint32_t shl_clamp(uint32_t x, uint32_t s) { return __funnelshift_lc(0u, x, s); }

// Rebuilds everything the chain left out from its entries {L_k, s'_k}, 32 entries per pass, all lanes in parallel.
// Entry k renormalises iff s'_k < 2^16.  The low end obeys  base_{k+1} = (base_k + L_k) << sh_k  (sh_k = 16 or 0,
// mod 2^32), a composition of maps  x -> (x << S) + A  which is closed under composition
// ((x << S1) + A1) << S2) + A2 = (x << (S1 + S2)) + (A1 << S2) + A2,  so a warp-wide scan over (A, S) gives every
// lane the base its entry was added to; the carry out of the 32-bit window is then `base_k + L_k` overflowing, the
// emitted word is the top half of that sum, and the word index is a prefix popcount of the renormalisation flags.
struct EncDrain {
  uint32_t dbase;   // base before the first entry of the next pass
  uint32_t cnt;     // words emitted so far
  uint32_t cb_cur;  // carry bits of word group (cnt >> 5) accumulated so far
  uint16_t* words;
  uint32_t* cbits;
  uint32_t cap;  // capacity in words (multiple of 32)
  bool overflowed;
  int lane;

  __device__ __forceinline__ void begin(const EncState& st, uint16_t* w, uint32_t* cb, uint32_t cap_, int lane_) {
    dbase = st.base;
    cnt = st.cnt;
    words = w;
    cbits = cb;
    cap = cap_;
    overflowed = false;
    lane = lane_;
    cb_cur = (st.cnt == 0) ? 0u : cb[st.cnt >> 5];
  }

  // Entries [0, n) of `ent`, n <= kPasses * 32.  The scans of the passes do not depend on each other (only the
  // final application of `dbase` does), so they are issued together and their shuffle latencies overlap.
  template <int kPasses>
  __device__ __forceinline__ void drain(const uint2* ent, int n) {
    uint32_t Lk[kPasses], Ak[kPasses], Sk[kPasses], rmask[kPasses];
#pragma unroll
    for (int p = 0; p < kPasses; ++p) {
      const int k = p * 32 + lane;
      const bool act = k < n;
      const uint2 me = ent[act ? k : 0];
      const bool rr = act && me.y < 65536u;
      rmask[p] = __ballot_sync(kFull, rr);
      Lk[p] = act ? me.x : 0u;
      uint32_t S = rr ? 16u : 0u;
      uint32_t A = Lk[p] << S;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {  // inclusive scan of the maps: lane l ends with f_l o ... o f_0
        const uint32_t Ap = __shfl_up_sync(kFull, A, d);
        const uint32_t Sp = __shfl_up_sync(kFull, S, d);
        if (lane >= d) {
          A = shl_clamp(Ap, S) + A;
          S = min(Sp + S, 32u);
        }
      }
      Ak[p] = A;
      Sk[p] = S;
    }
#pragma unroll
    for (int p = 0; p < kPasses; ++p) {
      if (p * 32 >= n) break;
      // exclusive prefix = the map of the entries before this lane's
      uint32_t Ax = __shfl_up_sync(kFull, Ak[p], 1);
      uint32_t Sx = __shfl_up_sync(kFull, Sk[p], 1);
      if (lane == 0) {
        Ax = 0u;
        Sx = 0u;
      }
      const uint32_t before = shl_clamp(dbase, Sx) + Ax;  // base this entry's L was added to
      const uint32_t nb = before + Lk[p];
      const bool carry = nb < before;                     // (inactive lanes: L = 0, never)
      const bool ren = (rmask[p] >> lane) & 1u;
      const uint32_t my_cnt = cnt + __popc(rmask[p] & ((1u << lane) - 1u));  // word count before this entry
      if (ren) {
        if (my_cnt < cap) words[my_cnt] = (uint16_t)(nb >> 16);
        else overflowed = true;
      }
      const uint32_t g0 = cnt >> 5;
      const uint32_t bit = 1u << (my_cnt & 31u);
      const uint32_t m0 = __reduce_or_sync(kFull, (carry && (my_cnt >> 5) == g0) ? bit : 0u);
      const uint32_t m1 = __reduce_or_sync(kFull, (carry && (my_cnt >> 5) != g0) ? bit : 0u);
      const uint32_t pass_end = cnt + __popc(rmask[p]);
      cb_cur |= m0;
      if ((pass_end >> 5) != g0) {
        if (lane == 0 && g0 < (cap >> 5)) cbits[g0] = cb_cur;
        cb_cur = m1;
      }
      cnt = pass_end;
      // base after the last entry of this pass
      dbase = shl_clamp(dbase, __shfl_sync(kFull, Sk[p], 31)) + __shfl_sync(kFull, Ak[p], 31);
    }
  }

  __device__ __forceinline__ void end(DevError* err, long long stream) {
    if ((cnt >> 5) < (cap >> 5)) {
      if (lane == 0) cbits[cnt >> 5] = cb_cur;
    } else {
      overflowed = true;
    }
    if (__any_sync(kFull, overflowed)) report(err, kErrCapacity, stream, cnt, cnt, cap);
  }
};

enum : int { kModeIndex = 1, kModeF32 = 2 };

struct EncParams {
  const int32_t* lookup;
  const int2* rows;
  int n_rows;
  int uniform_prec;        // > 0: every row has this precision
  int n_sms;
  int rot;                 // warp-role rotation of the CTAs of the second wave (see encode_kernel)
  const void* value;       // int32 or float [S, n]
  const int32_t* index;    // [S, n] or null
  const float* qoff;       // channel+f32: [n_rows] or null; index+f32: loc [S, n] or null
  const int32_t* coff;     // f32 modes: cdf_offset [n_rows]
  long long n;
  long long n_streams;
  EncState* state;
  uint16_t* words;
  uint32_t* cbits;
  long long cap;  // words per stream
  DevError* err;
};

// The gather of one pass of 32 symbols is split in two stages so that no global-memory latency is
// ever exposed to the (in-order) warp:
//   stage A, three passes ahead : the symbol itself (y / value, index, loc) and, in channel mode, the row
//                                 descriptor and the per-row offsets -- all independent loads;
//   stage B, current pass       : quantise, range-check, escape mapping, then the two table loads and the
//                                 operand records written to shared memory for the serial chain.
struct Fetched {
  float y;
  int v;
  float loc_or_q;
  int coff;
  int row;
  int2 ri;
  bool valid;
};

struct Gathered {
  uint4 ops;       // pre-scaled operands (enc_operands)
  uint32_t prec;   // 0 = invalid / out of range
  uint32_t gamma;  // escape payload (0 = none)
  uint32_t sign;
};

template <int MODE>
__device__ __forceinline__ Fetched enc_fetch(const EncParams& P, long long s, long long j, uint32_t chan_row) {
  Fetched f;
  f.y = 0.f;
  f.v = 0;
  f.loc_or_q = 0.f;
  f.coff = 0;
  f.row = (int)chan_row;
  f.ri = make_int2(0, 0);
  f.valid = j < P.n;
  if (!f.valid) return f;
  const long long at = s * P.n + j;
  if (MODE & kModeF32) {
    f.y = __ldg(reinterpret_cast<const float*>(P.value) + at);
  } else {
    f.v = __ldg(reinterpret_cast<const int32_t*>(P.value) + at);
  }
  if (MODE & kModeIndex) {
    f.row = __ldg(P.index + at);
    if ((MODE & kModeF32) && P.qoff) f.loc_or_q = __ldg(P.qoff + at);
  } else {
    f.ri = __ldg(P.rows + f.row);
    if (MODE & kModeF32) {
      if (P.qoff) f.loc_or_q = __ldg(P.qoff + f.row);
      f.coff = __ldg(P.coff + f.row);
    }
  }
  return f;
}

template <int MODE>
__device__ __forceinline__ Gathered enc_gather(const EncParams& P, long long s, long long j, Fetched f) {
  Gathered g;
  g.ops = make_uint4(0u, 0u, 0u, 0u);
  g.prec = 0;
  g.gamma = 0;
  g.sign = 0;
  if (!f.valid) return g;
  if (MODE & kModeIndex) {
    if (f.row < 0 || f.row >= P.n_rows) {
      report(P.err, kErrIndex, s, j, f.row, P.n_rows);
      return g;
    }
    f.ri = __ldg(P.rows + f.row);
    if (MODE & kModeF32) f.coff = __ldg(P.coff + f.row);
  }
  int v = f.v;
  if (MODE & kModeF32) v = (int)rintf(f.y - f.loc_or_q) - f.coff;
  const int ncdf = row_ncdf(f.ri.y);
  if (!row_ovf(f.ri.y)) {
    if (v < 0 || v >= ncdf - 1) {
      report(P.err, kErrValue, s, j, v, ncdf - 1);
      return g;
    }
  } else {
    const int esc = ncdf - 2;
    if (v < 0) {
      g.gamma = (uint32_t)(-(long long)v);
      g.sign = 1;
      v = esc;
    } else if (v >= esc) {
      g.gamma = (uint32_t)(v - esc + 1);
      v = esc;
    }
  }
  const uint32_t lower = (uint32_t)__ldg(P.lookup + f.ri.x + v);
  const uint32_t upper = (uint32_t)__ldg(P.lookup + f.ri.x + v + 1);
  g.prec = (uint32_t)row_prec(f.ri.y);
  g.ops = enc_operands(lower, upper, g.prec);
  return g;
}

// Named barriers (bar.sync / bar.arrive) for the warp-to-warp hand-offs.
__device__ __forceinline__ void bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void bar_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// Shared state of one code stream's CTA.  The unit of every hand-off is a BLOCK of up to kBlock operand records
// (gather -> chain) and the same number of entries (chain -> drain), double buffered; one barrier round trip per
// block and direction.  The gather warp writes the record stream the chain consumes blindly: an escaping symbol
// is followed by the records of its Elias-gamma bits (OverflowEncode, range_coder_kernels.cc:306-321), so the
// chain warp has no special cases at all.
#ifndef TFCB_ENC_BLOCK
#define TFCB_ENC_BLOCK 256
#endif
constexpr int kBlock = TFCB_ENC_BLOCK;

struct BlockInfo {
  uint32_t n;     // records / entries in this block (kBlock except for the last one)
  uint32_t last;  // nonzero: no further block follows
};

struct EncShared {
  uint4 ops[2][kBlock + 2];   // (+2: the chain's operand prefetch may run two records past the block)
  uint2 ent[2][kBlock];
  BlockInfo ops_info[2];
  BlockInfo ent_info[2];
};

enum : int { kBarOpsFull = 1, kBarOpsEmpty = 3, kBarEntFull = 5, kBarEntEmpty = 7 };

// Gather-warp helper: appends records to the block stream, handing full blocks to the chain warp.
struct RecordWriter {
  EncShared* sh;
  long long blocks;  // blocks published so far
  int fill;          // records in the current block

  __device__ __forceinline__ void begin(EncShared* sh_) {
    sh = sh_;
    blocks = 0;
    fill = 0;
  }
  __device__ __forceinline__ uint4* cur() { return sh->ops[blocks & 1]; }
  __device__ __forceinline__ void publish(bool last) {
    const int b = (int)(blocks & 1);
    if ((threadIdx.x & 31) == 0) {
      BlockInfo bi;
      bi.n = (uint32_t)fill;
      bi.last = last ? 1u : 0u;
      sh->ops_info[b] = bi;
    }
    bar_arrive(kBarOpsFull + b, 64);  // arrive orders the preceding shared-memory writes
    ++blocks;
    fill = 0;
    if (!last && blocks >= 2) bar_sync(kBarOpsEmpty + (int)(blocks & 1), 64);  // the chain is done with that buffer
  }
  // Appends this pass's records: lane's own record `first` at pass-local position `pre`, followed by `extra` more
  // produced by `rec(i)`; `total` = all lanes' records.  Blocks are filled exactly; a pass may straddle blocks.
  template <typename F>
  __device__ __forceinline__ void append(uint4 first, int pre, int extra, int total, bool has, F rec) {
    int done = 0;
    while (done < total) {
      const int room = kBlock - fill;
      const int take = min(room, total - done);
      uint4* dst = cur() + fill - done;  // record with pass-local position i goes to dst[i]
      if (has) {
        if (pre >= done && pre < done + take) dst[pre] = first;
        for (int i = 0; i < extra; ++i) {
          const int at = pre + 1 + i;
          if (at >= done && at < done + take) dst[at] = rec(i);
        }
      }
      fill += take;
      done += take;
      if (fill == kBlock) publish(false);
    }
  }
};

// Record i of the escape tail of OverflowEncode (range_coder_kernels.cc:306-321): nb - 1 zero bits, the nb bits
// of g (MSB first), then the sign, each coded with the uniform binary CDF {0, 1, 2} at precision 1.
__device__ __forceinline__ uint4 gamma_record(uint32_t g, uint32_t sign, int nb, int i) {
  uint32_t bit;
  if (i < nb - 1) bit = 0u;
  else if (i < 2 * nb - 1) bit = (g >> (2 * nb - 2 - i)) & 1u;
  else bit = sign;
  return enc_operands(bit, bit + 1u, 1u);
}

template <int MODE>
__global__ void __launch_bounds__(192) encode_kernel(const EncParams P) {
  __shared__ __align__(16) EncShared sh;
  const long long s = blockIdx.x;
  const int lane = threadIdx.x & 31;
  // Roles: 0 chain, 1 gather, 2 drain, 3 idle (exits at once).  Only the per-stream latency of the chain warp
  // matters (there are more schedulers than streams), so the layout's job is to keep a chain warp alone on its
  // sub-partition (warp slot mod 4) when two CTAs share an SM:
  //   six warps per CTA (P.rot < 0): warp 0 chain, 1 gather, 5 drain, 2..4 idle -- the first CTA of an SM takes slots
  //     0..5 (chain on sub-partition 0, gather + drain on 1), the second slots 6..11 (chain on 2, gather + drain on 3);
  //   four warps per CTA (P.rot = 0..3): roles rotated by P.rot in the CTAs launched after the first wave.
  // Measured: profiles/r2_encode_notes.md.
  const int warp = threadIdx.x >> 5;
  int role;
  if (P.rot < 0) {
    role = warp == 0 ? 0 : (warp == 1 ? 1 : (warp == 5 ? 2 : 3));
  } else {
    const int rot = (blockIdx.x >= (unsigned)P.n_sms) ? P.rot : 0;
    role = (warp - rot) & 3;
  }
  if (role == 3) return;

  if (role == 1) {
    // ------------------------------- gather warp -------------------------------
    uint32_t row_a = 0, chan_step = 0;
    if (!(MODE & kModeIndex)) {
      row_a = (uint32_t)lane % (uint32_t)P.n_rows;
      chan_step = 32u % (uint32_t)P.n_rows;
    }
    auto advance_row = [&]() {
      if (!(MODE & kModeIndex)) {
        row_a += chan_step;
        if (row_a >= (uint32_t)P.n_rows) row_a -= (uint32_t)P.n_rows;
      }
    };
    // stage A (symbol loads) runs three 32-symbol passes ahead of stage B: no global latency is waited for
    Fetched f0 = enc_fetch<MODE>(P, s, lane, row_a);
    advance_row();
    Fetched f1 = enc_fetch<MODE>(P, s, 32 + lane, row_a);
    advance_row();
    Fetched f2 = enc_fetch<MODE>(P, s, 64 + lane, row_a);
    advance_row();
    RecordWriter w;
    w.begin(&sh);
    const long long n_pass = (P.n + 31) / 32;
    bool stop = false;
    for (long long pass = 0; pass < n_pass && !stop; ++pass) {
      const Fetched fcur = f0;
      f0 = f1;
      f1 = f2;
      f2 = enc_fetch<MODE>(P, s, (pass + 3) * 32 + lane, row_a);
      advance_row();
      const long long j0 = pass * 32;
      const Gathered cur = enc_gather<MODE>(P, s, j0 + lane, fcur);
      const int count = (int)min(32ll, P.n - j0);
      const bool has = lane < count;
      const unsigned esc_mask = __ballot_sync(kFull, cur.gamma != 0);
      const unsigned bad_mask = __ballot_sync(kFull, cur.prec == 0 && has);
      if (bad_mask) {  // argument error already recorded: code nothing more of this stream
        stop = true;
        break;
      }
      if (esc_mask == 0) {
        if (w.fill + count <= kBlock) {  // the common case: one store per lane
          if (has) w.cur()[w.fill + lane] = cur.ops;
          w.fill += count;
          if (w.fill == kBlock) w.publish(false);
        } else {
          w.append(cur.ops, lane, 0, count, has, [&](int) { return cur.ops; });
        }
      } else {
        const int nb = cur.gamma ? 32 - __clz(cur.gamma) : 0;
        const int mine = has ? 1 + 2 * nb : 0;
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int t = __shfl_up_sync(kFull, incl, d);
          if (lane >= d) incl += t;
        }
        const int total = __shfl_sync(kFull, incl, 31);
        w.append(cur.ops, incl - mine, 2 * nb, total, has,
                 [&](int i) { return gamma_record(cur.gamma, cur.sign, nb, i); });
      }
    }
    w.publish(true);  // (possibly empty) final block: lets the other two warps finish
    return;
  }

  if (role == 2) {
    // ------------------------------- drain warp -------------------------------
    EncDrain d;
    d.begin(P.state[s], P.words + s * P.cap, P.cbits + s * (P.cap >> 5), (uint32_t)P.cap, lane);
    for (long long k = 0;; ++k) {
      const int b = (int)(k & 1);
      bar_sync(kBarEntFull + b, 64);
      const BlockInfo bi = sh.ent_info[b];
      d.drain<kBlock / 32>(sh.ent[b], (int)bi.n);
      if (bi.last) break;
      bar_arrive(kBarEntEmpty + b, 64);
    }
    d.end(P.err, s);
    if (lane == 0) {
      P.state[s].base = d.dbase;
      P.state[s].cnt = d.cnt;
    }
    return;
  }

  // --------------------------------- chain warp ---------------------------------
  EncChain c;
  c.s = P.state[s].raw;
  for (long long k = 0;; ++k) {
    const int b = (int)(k & 1);
    bar_sync(kBarOpsFull + b, 64);
    const BlockInfo bi = sh.ops_info[b];
    if (k >= 2) bar_sync(kBarEntEmpty + b, 64);  // the drain warp is done with this entry buffer
    // operands are fetched two records ahead so that the shared-memory latency stays off the chain; two 64-bit
    // loads per record: each multiply-add gets its addend in a register pair of its own
    const uint2* q = reinterpret_cast<const uint2*>(sh.ops[b]);
    uint2* e = sh.ent[b];
    const int n = (int)bi.n;
    int kk = 0;
    uint2 l0 = q[0], h0 = q[1], l1 = q[2], h1 = q[3];
#pragma unroll 1
    for (; kk + 8 <= n; kk += 8) {
      const uint2* p = q + 2 * kk;
      uint2* const eo = e + kk;
#pragma unroll
      for (int j = 0; j < 8; j += 2) {  // immediates only
        const uint2 a0 = l0, b0 = h0, a1 = l1, b1 = h1;
        l0 = p[2 * j + 4];
        h0 = p[2 * j + 5];
        l1 = p[2 * j + 6];
        h1 = p[2 * j + 7];
        eo[j] = c.step(a0, b0);
        eo[j + 1] = c.step(a1, b1);
      }
    }
    for (; kk < n; ++kk) e[kk] = c.step(sh.ops[b][kk]);
    if (lane == 0) sh.ent_info[b] = bi;
    bar_arrive(kBarEntFull + b, 64);  // arrive orders the preceding shared-memory writes
    if (bi.last) break;
    bar_arrive(kBarOpsEmpty + b, 64);
  }
  if (lane == 0) {
    P.state[s].span = (c.s < 65536u) ? ((c.s << 16) | 0xFFFFu) : c.s;
    P.state[s].raw = c.s;
  }
}

// ---------------------------------------------------------------------------------------------
// Encoder finalize
// ---------------------------------------------------------------------------------------------
__global__ void enc_init_state_kernel(EncState* st, long long n) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) {
    EncState s;
    s.base = 0;
    s.span = 0xFFFFFFFFu;
    s.cnt = 0;
    s.raw = 0xFFFFFFFFu;
    st[i] = s;
  }
}

// Tail rule of RangeEncoder::Finalize (range_coder.cc:266-307) expressed on (words, state).
// Returns the string length; `straddle` = the interval still contains 2^32 ("state 1").
__device__ __forceinline__ long long enc_final_length(const EncState& st, const uint16_t* words,
                                                      bool* straddle, uint32_t* tail, int* ntail) {
  const uint32_t top_end = st.base + st.span;
  *ntail = 0;
  *tail = 0;
  if (top_end < st.base) {
    // The reference picks 2^32: +1 ripples through the run of 0xFFFF words left of the window into
    // word d (the delayed word, < 0xFFFF); everything right of d becomes zero and is dropped, and so
    // is the low byte of word d when it is zero.
    *straddle = true;
    uint32_t d = st.cnt - 1u;
    while (d > 0 && words[d] == 0xFFFFu) --d;
    const uint32_t wd = ((uint32_t)words[d] + 1u) & 0xFFFFu;
    return 2ll * d + 1 + ((wd & 0xFFu) ? 1 : 0);
  }
  *straddle = false;
  if (st.base != 0) {
    const uint32_t r24 = ((st.base - 1u) >> 24) + 1u;
    if (r24 <= (top_end >> 24)) {
      *tail = r24 << 8;
      *ntail = 1;
    } else {
      const uint32_t r16 = ((st.base - 1u) >> 16) + 1u;
      *tail = r16;
      *ntail = (r16 & 0xFFu) ? 2 : 1;
    }
  }
  return 2ll * st.cnt + *ntail;
}

__global__ void enc_lengths_kernel(const EncState* state, const uint16_t* words, long long cap,
                                   long long n_streams, long long* lens) {
  const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (s >= n_streams) return;
  bool straddle;
  uint32_t tail;
  int ntail;
  lens[s] = enc_final_length(state[s], words + s * cap, &straddle, &tail, &ntail);
}

// Single-block exclusive scan: offsets[0..n] from lens[0..n-1].
__global__ void exclusive_scan_kernel(const long long* lens, long long n, long long* offsets) {
  __shared__ long long warp_sums[32];
  __shared__ long long carry_s;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (long long base = 0; base < n; base += blockDim.x) {
    const long long i = base + tid;
    long long v = (i < n) ? lens[i] : 0;
    long long x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const long long y = __shfl_up_sync(kFull, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
      long long w = (lane < (int)(blockDim.x >> 5)) ? warp_sums[lane] : 0;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const long long y = __shfl_up_sync(kFull, w, d);
        if (lane >= d) w += y;
      }
      warp_sums[lane] = w;  // inclusive
    }
    __syncthreads();
    const long long before = carry_s + (wid ? warp_sums[wid - 1] : 0) + (x - v);
    if (i < n) offsets[i] = before;
    __syncthreads();
    if (tid == blockDim.x - 1) carry_s = before + v;
    __syncthreads();
  }
  if (tid == 0) offsets[n] = carry_s;
}

// One warp per stream: resolve carries right-to-left, 32 words per step, and write the bytes.
// One CTA of kWriteWarps warps per stream.  The carry chain runs right to left over 32-word groups; it is cut into
// kWriteWarps segments: every warp first runs its segment's chain for BOTH possible carries entering it (two adds per
// group instead of one), the segments' carry-ins are then resolved through shared memory (a chain of kWriteWarps
// steps), and each warp resolves and writes its own segment.  (One warp per stream walked 200 groups serially:
// 46 us of the 714 us cfg2 step.)
constexpr int kWriteWarps = 8;

__global__ void __launch_bounds__(32 * kWriteWarps) enc_write_kernel(const EncState* state, const uint16_t* words,
                                                                    const uint32_t* cbits, long long cap,
                                                                    long long n_streams,
                                                                    const long long* offsets, uint8_t* out) {
  __shared__ uint32_t seg_out[kWriteWarps][2];
  const long long s = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (s >= n_streams) return;
  const EncState st = state[s];
  const uint16_t* w = words + s * cap;
  const uint32_t* cb = cbits + s * (cap >> 5);
  uint8_t* dst = out + offsets[s];
  bool straddle;
  uint32_t tail;
  int ntail;
  const long long len = enc_final_length(st, w, &straddle, &tail, &ntail);
  const long long body = straddle ? len : 2ll * st.cnt;  // bytes that come from resolved words

  const long long n_groups = ((long long)st.cnt + 31) >> 5;
  const long long per = (n_groups + kWriteWarps - 1) / kWriteWarps;
  const long long g_lo = min((long long)warp * per, n_groups), g_hi = min(g_lo + per, n_groups);  // this warp's groups
  const bool even = ((reinterpret_cast<uintptr_t>(dst)) & 1) == 0;
  constexpr int kBatch = 8;  // groups whose (independent) loads are in flight together

  // One pass over the segment [g_lo, g_hi), right to left.  WRITE = false: only the carries leaving the segment for a
  // carry of 0 and of 1 entering it; WRITE = true: resolve with the real carry `x0` and store the bytes.
  auto pass = [&](uint32_t& x0, uint32_t& x1, const bool write) {
    for (long long gt = g_hi; gt > g_lo; gt -= kBatch) {
      uint32_t word[kBatch], F[kBatch];
#pragma unroll
      for (int i = 0; i < kBatch; ++i) {
        const long long g = gt - 1 - i;
        const uint32_t idx = (uint32_t)(g << 5) + lane;
        word[i] = (g >= g_lo && idx < st.cnt) ? (uint32_t)w[idx] : 0u;
        F[i] = (g >= g_lo) ? cb[g] : 0u;
      }
#pragma unroll
      for (int i = 0; i < kBatch; ++i) {
        const long long g = gt - 1 - i;
        if (g < g_lo) break;
        const uint32_t idx = (uint32_t)(g << 5) + lane;
        const bool live = idx < st.cnt;
        uint32_t Fm = F[i];
        const uint32_t fill = st.cnt - (uint32_t)(g << 5);
        if (fill < 32u) Fm &= (1u << fill) - 1u;
        // P: word propagates a carry.  Dead lanes right of the last word must pass the carry through.
        const uint32_t Pm = __ballot_sync(kFull, live ? (word[i] == 0xFFFFu) : true);
        // position j = 31 - lane (bit 0 = right-most word); c[j+1] = F[31-j] | (P[31-j] & c[j])
        const uint32_t G = __brev(Fm);
        const uint32_t A = G | __brev(Pm);
        const unsigned long long sum = (unsigned long long)A + G + x0;
        if (!write) x1 = (uint32_t)(((unsigned long long)A + G + x1) >> 32) & 1u;
        const uint32_t cin = (uint32_t)sum ^ A ^ G;  // bit j = carry into position j
        const uint32_t my_c = (cin >> (31 - lane)) & 1u;
        x0 = (uint32_t)(sum >> 32) & 1u;
        if (write && live) {
          const uint32_t r = (word[i] + my_c) & 0xFFFFu;
          const long long b0 = 2ll * idx;
          if (even && b0 + 1 < body) {
            *reinterpret_cast<uint16_t*>(dst + b0) = (uint16_t)((r >> 8) | ((r & 0xFFu) << 8));  // big endian
          } else {
            if (b0 < body) dst[b0] = (uint8_t)(r >> 8);
            if (b0 + 1 < body) dst[b0 + 1] = (uint8_t)r;
          }
        }
      }
    }
  };
  uint32_t o0 = 0u, o1 = 1u;
  pass(o0, o1, false);
  if (lane == 0) {
    seg_out[warp][0] = o0;
    seg_out[warp][1] = o1;
  }
  __syncthreads();
  // carry entering the right-most word (index cnt - 1), then through the segments to the right of this one
  uint32_t x = straddle ? 1u : ((cb[st.cnt >> 5] >> (st.cnt & 31u)) & 1u);
  for (int k = kWriteWarps - 1; k > warp; --k) x = seg_out[k][x];
  uint32_t unused = 0u;
  pass(x, unused, true);
  if (!straddle && threadIdx.x == 0) {
    if (ntail >= 1) dst[body] = (uint8_t)(tail >> 8);
    if (ntail == 2) dst[body + 1] = (uint8_t)tail;
  }
}

__global__ void enc_grow_kernel(const uint16_t* src, const uint32_t* src_cb, long long src_cap,
                                uint16_t* dst, uint32_t* dst_cb, long long dst_cap,
                                const EncState* state) {
  const long long s = blockIdx.x;
  const uint32_t used = (state[s].cnt + 31u) & ~31u;
  for (uint32_t i = threadIdx.x; i < used; i += blockDim.x) dst[s * dst_cap + i] = src[s * src_cap + i];
  for (uint32_t i = threadIdx.x; i <= (state[s].cnt >> 5); i += blockDim.x)
    dst_cb[s * (dst_cap >> 5) + i] = src_cb[s * (src_cap >> 5) + i];
}

// ---------------------------------------------------------------------------------------------
// Decoder
// ---------------------------------------------------------------------------------------------
struct DecState {
  uint32_t base, span, value;
  uint32_t pos;  // 16-bit words consumed (starts at 2)
};

struct DecParams {
  const int32_t* lookup;
  const int2* rows;
  const uint2* pairs;
  const int4* rows4;
  int n_rows;
  long long lookup_len;
  long long n_pairs;
  int zero_win;
  const uint8_t* bytes;
  const long long* offsets;
  const int32_t* index;
  void* out;               // int32 or float [S, n]
  const float* qoff;       // channel: [n_rows]; index: loc [S, n]
  const int32_t* coff;     // [n_rows]
  long long n;
  long long n_streams;
  DecState* state;
  DevError* err;
};

struct ByteWindow {
  const uint8_t* p;
  long long len;
  uint32_t lane_word;  // word (pos & ~31) + lane
  uint32_t next;       // word at index pos
};

__device__ __forceinline__ uint32_t bw_fetch(const ByteWindow& w, long long word_idx) {
  const long long b = 2 * word_idx;
  uint32_t hi = 0, lo = 0;
  if (b < w.len) hi = w.p[b];
  if (b + 1 < w.len) lo = w.p[b + 1];
  return (hi << 8) | lo;
}

__device__ __forceinline__ void bw_seek(ByteWindow& w, uint32_t pos, int lane) {
  w.lane_word = bw_fetch(w, (long long)(pos & ~31u) + lane);
  w.next = __shfl_sync(kFull, w.lane_word, pos & 31u);
}

struct DecChain {
  uint32_t base, span, value, pos;
};

__device__ __forceinline__ void dec_update(DecChain& c, ByteWindow& w, uint32_t a, uint32_t b, int lane) {
  c.base += a;
  c.span = b - a - 1u;
  if (c.span < 65536u) {
    c.base <<= 16;
    c.span = (c.span << 16) | 0xFFFFu;
    c.value = (c.value << 16) | w.next;
    c.pos += 1;
    if ((c.pos & 31u) == 0) {
      bw_seek(w, c.pos, lane);
    } else {
      w.next = __shfl_sync(kFull, w.lane_word, c.pos & 31u);
    }
  }
}

// Smallest i in [1, ncdf-1] with scale(cdf[i]) > value - base; identical to the reference's binary
// search (range_coder.h:204-222,241-251) for every monotone CDF.  Clamped for corrupt streams.
__device__ __forceinline__ int dec_symbol(DecChain& c, ByteWindow& w, const int32_t* cdf, int ncdf,
                                          uint32_t p, int lane) {
  const uint32_t v = c.value - c.base;
  int lo_i = 1;
  int n = ncdf - 1;
  int i;
  for (;;) {
    const int stride = (n + 31) >> 5;
    int off = (lane + 1) * stride - 1;
    if (off > n - 1) off = n - 1;
    const uint32_t cv = (uint32_t)cdf[lo_i + off];
    const bool pred = v < scale_cum(c.span, cv, p);
    // scale_cum truncates 2^32 to 0; that only happens for cv == 2^p with span == 2^32-1, where the
    // true value 2^32 exceeds every v.
    const bool full = (cv == (1u << p)) && (c.span == 0xFFFFFFFFu);
    const unsigned m = __ballot_sync(kFull, pred || full);
    const int f = m ? (__ffs(m) - 1) : 31;
    if (stride == 1) {
      i = lo_i + min(f, n - 1);
      break;
    }
    const int skip = min(f * stride, n - 1);
    lo_i += skip;
    n = min(stride, n - skip);
  }
  const uint32_t ca = (uint32_t)cdf[i - 1];
  const uint32_t cb = (uint32_t)cdf[i];
  dec_update(c, w, scale_cum(c.span, ca, p), scale_cum(c.span, cb, p), lane);
  return i - 1;
}


// ---------------------------------------------------------------------------------------------
// Decoder: three warps per stream (prepare / chain / resolve), pre-scaled search keys
// ---------------------------------------------------------------------------------------------
// The decoder has the encoder's recurrence plus a search per symbol.  As in the encoder everything that
// is not the recurrence leaves the latency-critical warp:
//   prepare warp : per symbol the row's search window (64 pre-scaled keys around the row's median), and the
//                  stream's next 16-bit words in a shared-memory ring well ahead of the chain;
//   chain warp   : every lane evaluates two keys B'(c) = T(c) - 1 = hi32(span*c' + addend) (one IMAD.HI
//                  each), two warp reductions give the bracketing pair (a, b1) and the new interval; the
//                  SYMBOL INDEX is not needed to continue -- only {value - base, span} are recorded;
//   resolve warp : recovers the symbol index of 32 recorded symbols at a time by binary search over the
//                  window, applies cdf_offset / de-quantisation and writes the output coalesced.
// Rare cases (escape symbols, symbols outside the window, rows wider than the window) are handled on the
// chain warp by a generic warp-parallel search and hand the finished symbol to the resolve warp.
constexpr int kDecGroup = 128;
constexpr int kRing = 2048;       // words; the prepare warp keeps [pos, pos + kRingAhead) valid
constexpr int kRingAhead = 1536;  // > words two groups can consume even if every symbol escapes (256 * 5.1)

struct DecDesc {      // one symbol's search window, prepared ahead of the chain
  int win;            // key index of the window's first key (segment start + wfirst; the zero window if irregular)
  uint32_t thr;       // the window's answer needs a candidate below v unless it starts the row: slow if a < thr
  int seg;            // key index of cdf[0]
  int n;              // ncdf - 1, bit 31: overflow row
};

struct DecShared {
  DecDesc desc[2][kDecGroup + 2];
  uint2 ent[2][kDecGroup];        // {value - base, span} before the symbol's update
  int ovr[2][kDecGroup];          // symbols finished on the chain warp (escapes, window misses)
  unsigned ovr_mask[2][kDecGroup / 32];
  unsigned bad[2];
  unsigned count[2];
  unsigned rbad[2];    // chain -> resolve copies (the prepare warp may already be two groups ahead)
  unsigned rcount[2];
  unsigned pos_pub[2]; // chain -> prepare: stream position (16-bit words) after the group that used buffer b
};

enum : int { kBarDescFull = 1, kBarDescEmpty = 3, kBarDecEntFull = 5, kBarDecEntEmpty = 7 };

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t opaque(uint32_t x) {
  asm volatile("mov.u32 %0, %0;" : "+r"(x));
  return x;
}

__device__ __forceinline__ uint32_t key_bound(uint32_t span, uint2 q) {  // B'(c) = floor(size*c/2^p) - 1
  return (uint32_t)(((unsigned long long)span * q.x + (((unsigned long long)q.y << 32) | q.x)) >> 32);
}

__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
  uint2 r;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr));
  return r;
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
  uint32_t r;
  asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(addr));
  return r;
}

// volatile: keeps the interval update ahead of the branch that follows it in program order
__device__ __forceinline__ uint32_t prmt(uint32_t x, uint32_t y, uint32_t sel) {
  uint32_t r;
  asm volatile("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(y), "r"(sel));
  return r;
}

struct Dec2 {
  uint32_t base, span, value;
  uint32_t pos2;       // stream position in BYTES (2 * word index)
  uint32_t next;       // word at that position
  uint32_t ring_addr;  // shared address of the word ring (4096-byte aligned)
  int lane;

  __device__ __forceinline__ void seek() { next = lds_u16(ring_addr | (pos2 & (2 * kRing - 2))); }
  // new interval [base + a, base + b1] and 16-bit renormalisation (range_coder.h:255-268); branch free:
  // all three 16-bit shifts are one byte permute with a shared selector
  __device__ __forceinline__ void update(uint32_t a, uint32_t b1) {
    const uint32_t nb = base + a;
    const uint32_t s = b1 - a;
    const bool renorm = s < 65536u;
    const uint32_t sel = renorm ? 0x1054u : 0x3210u;  // {x.b1, x.b0, y.b1, y.b0} : x
    span = prmt(s, 0xFFFFFFFFu, sel);
    base = prmt(nb, 0u, sel);
    value = prmt(value, next, sel);
    pos2 += renorm ? 2u : 0u;
    next = lds_u16(ring_addr | (pos2 & (2 * kRing - 2)));  // consumed at the next renormalisation, not before
  }
  // DecodeLinearly({0,1,2}, 1), range_coder_kernels.cc:450,461-469
  __device__ __forceinline__ uint32_t bit() {
    const uint32_t v = value - base;
    const uint32_t half = key_bound(span, make_uint2(0x80000000u, 0u)) ;  // floor(size / 2) ... see below
    // key_bound with addend_hi = 0 returns hi32(span*c' + c') = floor(size * 1 / 2) exactly (no "-1")
    const uint32_t b = (v < half) ? 0u : 1u;
    update(b ? half : 0u, b ? span : half - 1u);
    return b;
  }
  // Generic warp-parallel search over the whole row (pairs[start .. start + n]); returns the symbol.
  __device__ __forceinline__ int search_row(const uint2* pairs, int start, int n, uint32_t* a_out, uint32_t* b_out) {
    const uint32_t v = value - base;
    int lo_i = 0, hi_i = n;
    for (;;) {
      const int len = hi_i - lo_i;
      const bool final_round = len <= 63;
      const int stride = final_round ? 1 : ((len + 63) >> 6);
      int i0, i1;
      if (final_round) {
        i0 = lo_i + lane;
        i1 = lo_i + lane + 32;
      } else {
        i0 = lo_i + (lane + 1) * stride;
        i1 = lo_i + (lane + 33) * stride;
      }
      i0 = min(i0, hi_i);
      i1 = min(i1, hi_i);
      const uint2 q0 = pairs[start + i0], q1 = pairs[start + i1];
      const uint32_t B0 = key_bound(span, q0), B1 = key_bound(span, q1);
      const bool ge0 = (v <= B0) && q0.x != 0u, ge1 = (v <= B1) && q1.x != 0u;
      // distinct candidates below v (clamped duplicates sit at hi_i, which is never below)
      const int below = __popc(__ballot_sync(kFull, !ge0)) + __popc(__ballot_sync(kFull, !ge1));
      if (final_round) {
        const uint32_t m = ge0 ? B0 : (ge1 ? B1 : 0xFFFFFFFFu);
        const uint32_t am = ge1 ? (ge0 ? 0u : B0 + 1u) : B1 + 1u;
        *b_out = __reduce_min_sync(kFull, m);
        *a_out = __reduce_max_sync(kFull, am);
        int i = lo_i + below;  // smallest index whose bound is >= v
        i = max(1, min(i, n));
        return i - 1;
      }
      const int f = min(below, 63);
      const int nlo = (f == 0) ? lo_i : min(lo_i + f * stride, hi_i - 1);
      const int nhi = min(lo_i + (f + 1) * stride, hi_i);
      lo_i = nlo;
      hi_i = max(nhi, nlo + 1);
    }
  }
};

template <int MODE, bool SMEM>
__global__ void __launch_bounds__(96) decode_kernel(const DecParams P) {
  extern __shared__ __align__(16) uint8_t s_dyn[];
  __shared__ __align__(16) DecShared sh;
  // The stream's next words, filled ahead by the prepare warp.  The chain warp addresses the ring as
  // base | offset, so its ABSOLUTE shared address must be 4096-byte aligned (static alignment is relative to the
  // CTA's window, which starts after the reserved 1 KB): carve an aligned ring out of a buffer twice the size.
  __shared__ __align__(16) uint16_t ring_buf[2 * kRing];
  uint16_t* const ring = ring_buf + (((4096u - (smem_addr(ring_buf) & 4095u)) & 4095u) >> 1);
  const long long s = blockIdx.x;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;  // 0 chain, 1 prepare, 2 resolve
  const long long n_groups = (P.n + kDecGroup - 1) / kDecGroup;

  // tables: shared memory when they fit (loaded by all three warps), global (L1/L2) otherwise
  const uint2* pairs = P.pairs;
  const int4* rows4 = P.rows4;
  if (SMEM) {
    uint2* sp = reinterpret_cast<uint2*>(s_dyn);
    int4* sr = reinterpret_cast<int4*>(s_dyn + ((P.n_pairs * 8 + 15) & ~15ll));
    for (int i = threadIdx.x; i < (int)P.n_pairs; i += blockDim.x) sp[i] = P.pairs[i];
    for (int i = threadIdx.x; i < P.n_rows; i += blockDim.x) sr[i] = P.rows4[i];
    __syncthreads();
    pairs = sp;
    rows4 = sr;
  }

  if (warp == 1) {
    // ------------------------------- prepare warp -------------------------------
    uint32_t chan_row = (uint32_t)lane % (uint32_t)P.n_rows;
    const uint32_t chan_step = 32u % (uint32_t)P.n_rows;
    ByteWindow bw;
    bw.p = P.bytes + P.offsets[s];
    bw.len = P.offsets[s + 1] - P.offsets[s];
    long long filled = (long long)P.state[s].pos;  // ring holds words [.., filled)
    auto fill_ring = [&](long long upto) {
      for (long long wi = filled + lane; wi < upto; wi += 32) ring[wi & (kRing - 1)] = (uint16_t)bw_fetch(bw, wi);
      filled = max(filled, upto);
    };
    fill_ring(filled + kRingAhead);
    for (long long g = 0; g < n_groups; ++g) {
      const int b = (int)(g & 1);
      if (g >= 2) {
        bar_sync(kBarDescEmpty + b, 64);
        fill_ring((long long)sh.pos_pub[b] + kRingAhead);  // pos after group g-2; two groups consume < kRingAhead
      }
      unsigned bad = 0;
#pragma unroll
      for (int sub = 0; sub < kDecGroup / 32; ++sub) {
        const long long j = g * kDecGroup + sub * 32 + lane;
        int row = (int)chan_row;
        if (MODE & kModeIndex) {
          row = 0;
          if (j < P.n) {
            row = __ldg(P.index + s * P.n + j);
            if (row < 0 || row >= P.n_rows) {
              report(P.err, kErrIndex, s, j, row, P.n_rows);
              row = -1;
            }
          }
          bad |= __ballot_sync(kFull, row < 0);
          if (row < 0) row = 0;
        } else {
          chan_row += chan_step;
          if (chan_row >= (uint32_t)P.n_rows) chan_row -= (uint32_t)P.n_rows;
        }
        const int4 r4 = rows4[row];
        DecDesc d;
        d.win = r4.w ? P.zero_win : r4.x + r4.z;
        d.thr = (r4.z > 1 || r4.w) ? 1u : 0u;
        d.seg = r4.x;
        d.n = (row_ncdf(r4.y) - 1) | (row_ovf(r4.y) ? (int)0x80000000 : 0);
        sh.desc[b][sub * 32 + lane] = d;
        if (sub == kDecGroup / 32 - 1 && lane < 2) sh.desc[b][kDecGroup + lane] = d;  // pipeline overrun slots
      }
      if (lane == 0) {
        sh.bad[b] = bad;
        sh.count[b] = (unsigned)min((long long)kDecGroup, P.n - g * kDecGroup);
      }
      bar_arrive(kBarDescFull + b, 64);
      if (bad) break;
    }
    return;
  }

  if (warp == 2) {
    // ------------------------------- resolve warp -------------------------------
    for (long long g = 0; g < n_groups; ++g) {
      const int b = (int)(g & 1);
      bar_sync(kBarDecEntFull + b, 64);
      const int count = (int)sh.rcount[b];
      if (sh.rbad[b]) break;
      for (int sub = 0; sub * 32 < count; ++sub) {
        const int k = sub * 32 + lane;
        const long long j = g * kDecGroup + k;
        if (k < count) {
          const long long at = s * P.n + j;
          int row;
          if (MODE & kModeIndex) row = __ldg(P.index + at);
          else row = (int)(j % P.n_rows);
          int sym;
          if ((sh.ovr_mask[b][sub] >> lane) & 1u) {
            sym = sh.ovr[b][k];
          } else {
            // binary search inside the window: smallest key index whose bound is >= v.  The key just left of
            // the window is known to be below (cdf[0] = 0, or a below-candidate existed), the last one >= v.
            const int4 r4 = rows4[row];
            const uint2 e = sh.ent[b][k];
            const uint2* keys = pairs + r4.x;
            int lo = r4.z - 1, hi = r4.z + 63;
#pragma unroll
            for (int it = 0; it < 6; ++it) {
              const int mid = (lo + hi + 1) >> 1;
              const bool ge = e.x <= key_bound(e.y, keys[mid]);
              hi = ge ? mid : hi;
              lo = ge ? lo : mid;
            }
            sym = hi - 1;
          }
          if (MODE & kModeF32) {
            float yv = (float)(sym + __ldg(P.coff + row));
            if (P.qoff) yv += (MODE & kModeIndex) ? __ldg(P.qoff + at) : __ldg(P.qoff + row);
            reinterpret_cast<float*>(P.out)[at] = yv;
          } else {
            reinterpret_cast<int32_t*>(P.out)[at] = sym;
          }
        }
      }
      if (g + 2 < n_groups) bar_arrive(kBarDecEntEmpty + b, 64);
    }
    return;
  }

  // --------------------------------- chain warp ---------------------------------
  Dec2 c;
  c.lane = lane;
  {
    const DecState st = P.state[s];
    c.base = st.base;
    c.span = st.span;
    c.value = st.value;
    c.pos2 = st.pos << 1;
  }
  c.ring_addr = opaque(smem_addr(ring));
  bool started = false;

  for (long long g = 0; g < n_groups; ++g) {
    const int b = (int)(g & 1);
    bar_sync(kBarDescFull + b, 64);
    if (!started) {  // the ring is valid from here on
      started = true;
      if (c.pos2 == 0) {  // fresh stream: the constructor reads four bytes (range_coder.h:79-83)
        c.value = ((uint32_t)ring[0] << 16) | (uint32_t)ring[1];
        c.pos2 = 4;
      }
      c.seek();
    }
    const bool bad = sh.bad[b] != 0;
    const int count = bad ? 0 : (int)sh.count[b];
    if (g >= 2) bar_sync(kBarDecEntEmpty + b, 64);  // the resolve warp is done with this entry buffer
    const DecDesc* desc = sh.desc[b];
    unsigned om0 = 0, om1 = 0, om2 = 0, om3 = 0;  // symbols finished on this warp (bit per symbol)
    // opaque shared addresses: keeps them in registers instead of being re-derived every symbol
    const uint32_t desc_addr = opaque(smem_addr(sh.desc[b]));
    const uint32_t ent_addr = opaque(smem_addr(sh.ent[b]));
    const uint2* lkeys = pairs + lane;  // this lane's two candidates: lkeys[win], lkeys[win + 32]
    const uint32_t lkeys_addr = SMEM ? opaque(smem_addr(lkeys)) : 0u;
    auto load_keys = [&](uint32_t win, uint2& q0, uint2& q1) {
      if (SMEM) {
        q0 = lds_v2(lkeys_addr + win * 8u);
        q1 = lds_v2(lkeys_addr + win * 8u + 256u);
      } else {
        q0 = __ldg(lkeys + win);
        q1 = __ldg(lkeys + win + 32);
      }
    };
    // One symbol of the fast path.  dc = descriptor of this symbol (reloaded with the one two ahead once
    // used), dn = the next symbol's; qc* = this symbol's candidate keys, qn* = receives the next symbol's.
    // Called with the roles swapped on alternate symbols so that the software pipeline needs no register
    // moves.  The interval update is issued BEFORE the "is this symbol special" branch so that the branch
    // latency is off the serial chain; a special symbol restores the state and leaves the loop.
    uint32_t daddr = desc_addr + 32u;  // descriptor two symbols ahead
    uint32_t eaddr = ent_addr;         // this symbol's entry
    const uint32_t eend = ent_addr + (uint32_t)count * 8u;
    uint32_t ra = 0, rb1 = 0, rthr = 0;  // the special symbol's window answer
    auto step = [&](uint2& dc, const uint2& dn, const uint2& qc0, const uint2& qc1, uint2& qn0, uint2& qn1) -> bool {
      load_keys(dn.x, qn0, qn1);
      const uint32_t thr = dc.y;
      dc = lds_v2(daddr);
      daddr += 16u;
      const uint32_t v = c.value - c.base;
      const uint32_t span0 = c.span;
      const uint32_t B0 = key_bound(span0, qc0), B1 = key_bound(span0, qc1);
      const bool ge0 = v <= B0, ge1 = v <= B1;
      const uint32_t m = ge0 ? B0 : (ge1 ? B1 : 0xFFFFFFFFu);
      const uint32_t am = ge1 ? (ge0 ? 0u : B0 + 1u) : B1 + 1u;
      const uint32_t b1 = __reduce_min_sync(kFull, m);
      const uint32_t a = __reduce_max_sync(kFull, am);
      sts_v2(eaddr, v, span0);
      eaddr += 8u;
      // Fast path: the window holds a key >= v that is not the row's last one, and (unless the window starts
      // the row) a key below v.  b1 >= span0 covers "no key" (~0) and the last bin (escape of overflow rows).
      const bool special = !(b1 < span0 && a >= thr);
      const uint32_t base0 = c.base, value0 = c.value, pos0 = c.pos2, next0 = c.next;
      c.update(a, b1);
      if (special) {
        c.base = base0;
        c.span = span0;
        c.value = value0;
        c.pos2 = pos0;
        c.next = next0;
        ra = a;
        rb1 = b1;
        rthr = thr;
      }
      return special;
    };
    uint2 da, db, qa0, qa1, qb0, qb1;
    auto prime = [&](uint32_t k) {  // restart the software pipeline at symbol k
      daddr = desc_addr + k * 16u;
      da = lds_v2(daddr);
      db = lds_v2(daddr + 16u);
      daddr += 32u;
      load_keys(da.x, qa0, qa1);
    };
    prime(0u);
    for (;;) {
      bool special = false;
      for (;;) {
        if (eaddr == eend) break;
        special = step(da, db, qa0, qa1, qb0, qb1);
        if (special) break;
        if (eaddr == eend) break;
        special = step(db, da, qb0, qb1, qa0, qa1);
        if (special) break;
      }
      if (!special) break;
      // ---- special symbol k: its entry is stored, the coder state is the one before it ----
      const int k = (int)((eaddr - 8u - ent_addr) >> 3);
      uint32_t a = ra, b1 = rb1;
      const DecDesc df = desc[k];
      const int n = df.n & 0x7FFFFFFF;
      const bool ovf = df.n < 0;
      const bool miss = (b1 == 0xFFFFFFFFu) || (a < rthr);
      int sym = n - 1;  // in-window hit with b1 == span: the row's last bin (regular rows)
      if (miss) sym = c.search_row(pairs, df.seg, n, &a, &b1);
      c.update(a, b1);
      bool finished = miss;
      if (ovf && sym == n - 1) {  // OverflowDecode, range_coder_kernels.cc:449-471
        int nb = 0;
        while (c.bit() == 0 && nb < 32) ++nb;  // valid int32 gamma codes have <= 31 zeros; bounds what a corrupt stream can consume (kRingAhead)
        uint32_t val = (nb < 32) ? (1u << nb) : 0u;
        int t = nb;
        while (--t >= 0) {
          const uint32_t bitv = c.bit();
          if (t < 32) val |= bitv << t;
        }
        const uint32_t sg = c.bit();
        sym = sg ? -(int)val : (int)val + (n - 1) - 1;
        finished = true;
      }
      if (finished) {  // otherwise the resolve warp finds the (last) bin like any other
        sh.ovr[b][k] = sym;
        const unsigned bitk = 1u << (k & 31);
        om0 |= (k >> 5) == 0 ? bitk : 0u;
        om1 |= (k >> 5) == 1 ? bitk : 0u;
        om2 |= (k >> 5) == 2 ? bitk : 0u;
        om3 |= (k >> 5) == 3 ? bitk : 0u;
      }
      prime((uint32_t)k + 1u);
    }

    const unsigned omask[kDecGroup / 32] = {om0, om1, om2, om3};
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < kDecGroup / 32; ++i) sh.ovr_mask[b][i] = omask[i];
      sh.rbad[b] = bad ? 1u : 0u;
      sh.rcount[b] = (unsigned)count;
    }
    bar_arrive(kBarDecEntFull + b, 64);
    if (bad) break;
    if (g + 2 < n_groups) {
      if (lane == 0) sh.pos_pub[b] = c.pos2 >> 1;
      bar_arrive(kBarDescEmpty + b, 64);
    }
  }
  if (lane == 0) {
    DecState st;
    st.base = c.base;
    st.span = c.span;
    st.value = c.value;
    st.pos = c.pos2 >> 1;
    P.state[s] = st;
  }
}

__global__ void dec_init_state_kernel(DecState* st, long long n) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) {
    DecState s;
    s.base = 0;
    s.span = 0xFFFFFFFFu;
    s.value = 0;
    s.pos = 0;
    st[i] = s;
  }
}

// RangeDecoder::Finalize, range_coder.h:144-169.
__global__ void dec_finalize_kernel(const DecState* state, const uint8_t* bytes, const long long* offsets,
                                    long long n, uint8_t* ok) {
  const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (s >= n) return;
  DecState st = state[s];
  const long long len = offsets[s + 1] - offsets[s];
  if (st.pos == 0) {  // never decoded from: only the constructor ran (four bytes, zero padded)
    const uint8_t* p = bytes + offsets[s];
    uint32_t v = 0;
    for (int i = 0; i < 4; ++i) v = (v << 8) | (i < len ? (uint32_t)p[i] : 0u);
    st.value = v;
    st.pos = 2;
  }
  bool good;
  if (2ll * st.pos < len) {
    good = false;  // did not read to the end
  } else {
    const uint32_t top_end = st.base + st.span;
    if (st.base == 0 || top_end < st.base) {
      good = (st.value == 0);
    } else {
      const int shift = (((st.base - 1u) >> 24) < (top_end >> 24)) ? 24 : 16;
      const uint32_t mid = ((st.base - 1u) >> shift) + 1u;
      good = ((mid << shift) == st.value);
    }
  }
  ok[s] = good ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------
// Legacy single-stream ops
// ---------------------------------------------------------------------------------------------
struct LegacyDims {
  int rank;               // merged rank (<= 6)
  long long data[6];      // merged data shape
  long long cdfd[6];      // merged cdf shape
  long long chip;         // strip length
};

__device__ __forceinline__ long long legacy_strip(const LegacyDims& d, long long lin) {
  long long off = 0, stride = d.chip;
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    if (i < d.rank) {
      const long long coord = lin % d.data[i];
      lin /= d.data[i];
      if (d.cdfd[i] > 1) off += coord * stride;
      stride *= d.cdfd[i];
    }
  }
  return off;
}

// CheckCdfValues, range_coding_kernels.cc:150-173.
__global__ void legacy_check_cdf_kernel(const int32_t* cdf, long long rows, long long size, int precision,
                                        DevError* err) {
  const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int32_t* s = cdf + r * size;
  const int32_t top = 1 << precision;
  if (s[0] != 0 || s[size - 1] != top) {
    report(err, kErrCdf, r, 0, s[0], s[size - 1], 1);
    return;
  }
  for (long long j = 0; j + 1 < size; ++j) {
    if (s[j + 1] <= s[j]) {
      report(err, kErrCdf, r, j, s[j], s[j + 1], 2);
      return;
    }
  }
}

__global__ void __launch_bounds__(32) legacy_encode_kernel(const int16_t* data, long long n,
                                                           const int32_t* cdf, LegacyDims dims,
                                                           int precision, int debug, EncState* state,
                                                           uint16_t* words, uint32_t* cbits,
                                                           long long cap, DevError* err) {
  __shared__ __align__(8) uint2 s_ent[32];
  const int lane = threadIdx.x;
  EncState st0;
  st0.base = 0;
  st0.span = 0xFFFFFFFFu;
  st0.cnt = 0;
  st0.raw = 0xFFFFFFFFu;
  EncChain c;
  c.s = st0.raw;
  EncDrain d;
  d.begin(st0, words, cbits, (uint32_t)cap, lane);
  for (long long g0 = 0; g0 < n; g0 += 32) {
    const int count = (int)min(32ll, n - g0);
    uint32_t lower = 0, upper = 1;
    bool bad = false;
    if (lane < count) {
      const long long j = g0 + lane;
      const long long v = data[j];
      if (v < 0 || dims.chip <= v + 1) {
        if (debug > 0) report(err, kErrValue, 0, j, v, dims.chip - 1);
        bad = true;  // without debug the reference has undefined behaviour; we stop instead
      } else {
        const int32_t* strip = cdf + legacy_strip(dims, j);
        lower = (uint32_t)strip[v];
        upper = (uint32_t)strip[v + 1];
        if (!(lower < upper) || upper > (1u << precision)) {
          bad = true;  // zero-probability symbol / invalid strip: UB in the reference
          report(err, kErrCdf, 0, j, lower, upper, 3);
        }
      }
    }
    if (__ballot_sync(kFull, bad)) break;
    uint2 mine = make_uint2(0u, 0u);
    for (int k = 0; k < count; ++k) {  // every lane runs the same recurrence; lane k keeps entry k
      const uint32_t lo = __shfl_sync(kFull, lower, k);
      const uint32_t hi = __shfl_sync(kFull, upper, k);
      const uint2 e = c.step(enc_operands(lo, hi, (uint32_t)precision));
      if (lane == k) mine = e;
    }
    s_ent[lane] = mine;
    __syncwarp();
    d.drain<1>(s_ent, count);
    __syncwarp();
  }
  d.end(err, 0);
  if (lane == 0) {
    EncState st;
    st.base = d.dbase;
    st.span = (c.s < 65536u) ? ((c.s << 16) | 0xFFFFu) : c.s;
    st.cnt = d.cnt;
    st.raw = c.s;
    state[0] = st;
  }
}

__global__ void __launch_bounds__(32) legacy_decode_kernel(const uint8_t* bytes, long long len,
                                                           long long n, const int32_t* cdf,
                                                           LegacyDims dims, int precision,
                                                           int16_t* out) {
  const int lane = threadIdx.x;
  DecChain c;
  c.base = 0;
  c.span = 0xFFFFFFFFu;
  ByteWindow w;
  w.p = bytes;
  w.len = len;
  c.value = (bw_fetch(w, 0) << 16) | bw_fetch(w, 1);
  c.pos = 2;
  bw_seek(w, c.pos, lane);
  for (long long g0 = 0; g0 < n; g0 += 32) {
    const int count = (int)min(32ll, n - g0);
    long long my_off = 0;
    if (lane < count) my_off = legacy_strip(dims, g0 + lane);
    int my_sym = 0;
    for (int k = 0; k < count; ++k) {
      const long long off = __shfl_sync(kFull, my_off, k);
      const int sym = dec_symbol(c, w, cdf + off, (int)dims.chip, (uint32_t)precision, lane);
      if (lane == k) my_sym = sym;
    }
    if (lane < count) out[g0 + lane] = (int16_t)my_sym;
  }
}

// ---------------------------------------------------------------------------------------------
// Host-side handles
// ---------------------------------------------------------------------------------------------

// ---------------------------------------------------------------------------------------------
// Device-table cache.  A model creates a handle per compress()/decompress() call with the same `lookup`
// every time (continuous_batched.py:381, :408): parsing and uploading it again (plus the stream
// synchronisation that keeps the host staging alive) would sit on the host's critical path of every step.
// Entries are keyed by content (hash, then full compare), pinned while a handle uses them, and evicted
// least-recently-used beyond kMaxEntries.  Uploads are complete (stream-synchronised) before an entry becomes
// visible, so any stream may use it.
// ---------------------------------------------------------------------------------------------
struct LookupCache {
  struct Entry {
    uint64_t hash = 0;
    int64_t cols = 0;
    bool for_decoder = false;
    int device = 0;
    int pins = 0;
    uint64_t last_use = 0;
    std::vector<int32_t> host;
    DeviceLookup lut;      // shallow copy of a cache entry's tables
  void* lut_token = nullptr;
  };
  static constexpr size_t kMaxEntries = 16;
  std::mutex mu;
  std::vector<Entry*> entries;
  uint64_t clock = 0;

  static uint64_t hash_of(const int32_t* p, int64_t n) {
    uint64_t hsh = 1469598103934665603ull;
    for (int64_t i = 0; i < n; ++i) hsh = (hsh ^ (uint32_t)p[i]) * 1099511628211ull;
    return hsh;
  }

  int acquire(const int32_t* host, int64_t len, int64_t cols, bool for_decoder, cudaStream_t s, DeviceLookup* out,
              void** token) {
    *token = nullptr;
    if (len < 0 || (len > 0 && !host)) return fail(TFCB_INVALID_ARGUMENT, "bad lookup table");
    int device = 0;
    cudaGetDevice(&device);
    const uint64_t hsh = hash_of(host, len);
    std::lock_guard<std::mutex> lock(mu);
    for (Entry* e : entries) {
      if (e->hash == hsh && e->cols == cols && e->for_decoder == for_decoder && e->device == device &&
          (int64_t)e->host.size() == len && (len == 0 || std::memcmp(e->host.data(), host, len * sizeof(int32_t)) == 0)) {
        e->pins++;
        e->last_use = ++clock;
        *out = e->lut;
        *token = e;
        return TFCB_OK;
      }
    }
    Entry* e = new Entry;
    int rc = e->lut.upload(host, len, cols, s, for_decoder);  // synchronises s: the tables are resident on return
    if (rc != TFCB_OK) {
      e->lut.release(s);
      delete e;
      return rc;
    }
    e->hash = hsh;
    e->cols = cols;
    e->for_decoder = for_decoder;
    e->device = device;
    e->pins = 1;
    e->last_use = ++clock;
    e->host.assign(host, host + len);
    entries.push_back(e);
    while (entries.size() > kMaxEntries) {
      size_t victim = entries.size();
      for (size_t i = 0; i < entries.size(); ++i)
        if (entries[i]->pins == 0 && (victim == entries.size() || entries[i]->last_use < entries[victim]->last_use)) victim = i;
      if (victim == entries.size()) break;  // everything is in use
      cudaDeviceSynchronize();  // rare (> kMaxEntries distinct tables): no kernel of any stream may still read it
      entries[victim]->lut.release(s);
      delete entries[victim];
      entries.erase(entries.begin() + victim);
    }
    *out = e->lut;
    *token = e;
    return TFCB_OK;
  }

  void release(void* token) {
    if (!token) return;
    std::lock_guard<std::mutex> lock(mu);
    static_cast<Entry*>(token)->pins--;
  }
};

LookupCache& lookup_cache() {
  static LookupCache* c = new LookupCache;  // leaked on purpose: no destructor order problems at exit
  return *c;
}

// Small pinned scratch per host thread for the device -> host words read at finalize.
void* pinned_scratch() {
  thread_local void* p = nullptr;
  if (!p) {
    if (cudaHostAlloc(&p, 256, cudaHostAllocDefault) != cudaSuccess) {
      (void)cudaGetLastError();
      p = nullptr;
    }
  }
  return p;
}

int decode_error(const DevError& e, const char* what);

int fetch_error(DevError* d_err, cudaStream_t s, const char* what) {
  DevError e;
  TFCB_CUDA_TRY(cudaMemcpyAsync(&e, d_err, sizeof e, cudaMemcpyDeviceToHost, s));
  TFCB_CUDA_TRY(cudaStreamSynchronize(s));
  return decode_error(e, what);
}

int decode_error(const DevError& e, const char* what) {
  switch (e.code) {
    case kErrNone:
      return TFCB_OK;
    case kErrIndex:
      return fail(TFCB_INVALID_ARGUMENT, "index=%lld not in range [0, %lld) (stream %lld, element %lld)",
                  e.value, e.limit, e.stream, e.pos);
    case kErrValue:
      if (std::strcmp(what, "legacy") == 0)
        return fail(TFCB_INVALID_ARGUMENT, "'data' value not in [0, %lld): value=%lld", e.limit, e.value);
      return fail(TFCB_INVALID_ARGUMENT, "value=%lld not in range [0, %lld) (stream %lld, element %lld)",
                  e.value, e.limit, e.stream, e.pos);
    case kErrCapacity:
      return fail(TFCB_CUDA_ERROR, "internal: output arena too small (stream %lld needs > %lld words)",
                  e.stream, e.limit);
    case kErrCdf:
      if (e.aux == 1)
        return fail(TFCB_INVALID_ARGUMENT, "CDF should start from 0 and end at 2^precision: cdf[0]=%lld, cdf[^1]=%lld",
                    e.value, e.limit);
      if (e.aux == 2) return fail(TFCB_INVALID_ARGUMENT, "CDF is not monotonic");
      return fail(TFCB_INVALID_ARGUMENT,
                  "symbol with zero probability or invalid CDF strip at element %lld: lower=%lld upper=%lld",
                  e.pos, e.value, e.limit);
  }
  return fail(TFCB_CUDA_ERROR, "unknown device error %d", e.code);
}

}  // namespace
}  // namespace tfcb

using namespace tfcb;

struct tfcb_encoder {
  DeviceLookup lut;      // shallow copy of a cache entry's tables
  void* lut_token = nullptr;
  long long n_streams = 0;
  EncState* state = nullptr;
  uint16_t* words = nullptr;
  uint32_t* cbits = nullptr;
  long long cap = 0;    // words per stream (multiple of 32)
  long long bound = 0;  // worst-case words emitted so far per stream
  DevError* err = nullptr;
  long long* lens = nullptr;
  long long* offsets = nullptr;
  uint8_t* out = nullptr;
  long long total = 0;
  bool finalized = false;
  cudaStream_t home = nullptr;
};

namespace {

// Worst-case 16-bit words one call can append per stream: every Encode(.., p) shrinks the interval by
// at most 2^p, i.e. consumes at most p bits; an escape adds at most 65 one-bit symbols.
long long words_bound(const tfcb_encoder* h, long long n) {
  const long long bits = h->lut.max_prec + (h->lut.any_overflow ? 65 : 0);
  return (n * bits + 15) / 16 + 2;
}

int ensure_capacity(tfcb_encoder* h, long long extra_words, cudaStream_t s) {
  const long long need = h->bound + extra_words + 32;
  if (need <= h->cap) return TFCB_OK;
  if (need >= (1ll << 31) - 64)
    return fail(TFCB_INVALID_ARGUMENT, "a single code stream may not exceed 2^31 16-bit words");
  const long long new_cap = (std::max(need, h->cap * 2) + 31) & ~31ll;
  uint16_t* nw = nullptr;
  uint32_t* nc = nullptr;
  const long long S = std::max<long long>(h->n_streams, 1);
  TFCB_TRY(dev_alloc((void**)&nw, (size_t)S * new_cap * sizeof(uint16_t), s));
  TFCB_TRY(dev_alloc((void**)&nc, (size_t)S * (new_cap >> 5) * sizeof(uint32_t), s));
  if (h->cap > 0 && h->bound > 0 && h->n_streams > 0) {
    enc_grow_kernel<<<(unsigned)h->n_streams, 128, 0, s>>>(h->words, h->cbits, h->cap, nw, nc, new_cap,
                                                           h->state);
    TFCB_LAUNCHED();
    TFCB_CUDA_TRY(cudaGetLastError());
  }
  dev_free(h->words, s);
  dev_free(h->cbits, s);
  h->words = nw;
  h->cbits = nc;
  h->cap = new_cap;
  return TFCB_OK;
}

// Warp-role rotation of the second-wave CTAs (0..3); TFCB_ENC_ROT overrides the default for experiments.
int enc_role_rotation() {
  static int rot = [] {
    const char* e = getenv("TFCB_ENC_ROT");
    if (e && e[0] >= '0' && e[0] <= '3') return e[0] - '0';
    return -1;  // default: the six-warp layout (11.7 vs 11.2 Gsym/s at cfg2, profiles/r2_encode_notes.md)
  }();
  return rot;
}

template <int MODE>
int launch_encode(tfcb_encoder* h, const void* value, const int32_t* index, const float* qoff,
                  const int32_t* coff, long long n, cudaStream_t s) {
  if (h->finalized) return fail(TFCB_INVALID_ARGUMENT, "encoder handle was already finalized");
  if (n < 0) return fail(TFCB_INVALID_ARGUMENT, "negative element count");
  if (h->n_streams == 0 || n == 0) return TFCB_OK;
  if (h->lut.n_rows == 0) return fail(TFCB_INVALID_ARGUMENT, "index=0 not in range [0, 0)");
  if (value == nullptr) return fail(TFCB_INVALID_ARGUMENT, "`value` is null");
  if ((MODE & kModeIndex) && index == nullptr) return fail(TFCB_INVALID_ARGUMENT, "`index` is null");
  if ((MODE & kModeF32) && coff == nullptr) return fail(TFCB_INVALID_ARGUMENT, "`cdf_offset` is null");
  const long long extra = words_bound(h, n);
  TFCB_TRY(ensure_capacity(h, extra, s));
  h->bound += extra;
  EncParams P;
  P.lookup = h->lut.lookup;
  P.rows = h->lut.rows;
  P.n_rows = h->lut.n_rows;
  P.uniform_prec = h->lut.uniform_prec;
  P.n_sms = device_sm_count();
  P.rot = enc_role_rotation();
  P.value = value;
  P.index = index;
  P.qoff = qoff;
  P.coff = coff;
  P.n = n;
  P.n_streams = h->n_streams;
  P.state = h->state;
  P.words = h->words;
  P.cbits = h->cbits;
  P.cap = h->cap;
  P.err = h->err;
  if (h->n_streams > 0x7FFFFFFFll) return fail(TFCB_INVALID_ARGUMENT, "too many streams");
  encode_kernel<MODE><<<(unsigned)h->n_streams, P.rot < 0 ? 192 : 128, 0, s>>>(P);
  TFCB_LAUNCHED();
  TFCB_CUDA_TRY(cudaGetLastError());
  return TFCB_OK;
}

}  // namespace

extern "C" {

int tfcb_encoder_create(const int32_t* lookup_host, int64_t lookup_len, int64_t lookup_cols,
                        int64_t n_streams, void* stream, tfcb_encoder** out) {
  if (!out) return fail(TFCB_INVALID_ARGUMENT, "null output handle");
  *out = nullptr;
  if (n_streams < 0) return fail(TFCB_INVALID_ARGUMENT, "negative stream count");
  cudaStream_t s = as_stream(stream);
  tfcb_encoder* h = new tfcb_encoder;
  h->home = s;
  h->n_streams = n_streams;
  int rc = lookup_cache().acquire(lookup_host, lookup_len, lookup_cols, /*for_decoder=*/false, s, &h->lut, &h->lut_token);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&h->state, std::max<int64_t>(n_streams, 1) * sizeof(EncState), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&h->err, sizeof(DevError), s);
  if (rc != TFCB_OK) {
    tfcb_encoder_destroy(h);
    return rc;
  }
  cudaMemsetAsync(h->err, 0, sizeof(DevError), s);
  if (n_streams > 0) {
    enc_init_state_kernel<<<(unsigned)((n_streams + 255) / 256), 256, 0, s>>>(h->state, n_streams);
    TFCB_LAUNCHED();
  }
  if (cudaGetLastError() != cudaSuccess) {
    tfcb_encoder_destroy(h);
    return fail(TFCB_CUDA_ERROR, "encoder state initialisation failed");
  }
  *out = h;
  return TFCB_OK;
}

int tfcb_encode_channel(tfcb_encoder* h, const int32_t* value_dev, int64_t n, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not an encoder");
  return launch_encode<0>(h, value_dev, nullptr, nullptr, nullptr, n, as_stream(stream));
}

int tfcb_encode_index(tfcb_encoder* h, const int32_t* index_dev, const int32_t* value_dev, int64_t n,
                      void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not an encoder");
  return launch_encode<kModeIndex>(h, value_dev, index_dev, nullptr, nullptr, n, as_stream(stream));
}

int tfcb_encode_channel_f32(tfcb_encoder* h, const float* y_dev, const float* quant_offset_dev,
                            const int32_t* cdf_offset_dev, int64_t n, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not an encoder");
  return launch_encode<kModeF32>(h, y_dev, nullptr, quant_offset_dev, cdf_offset_dev, n, as_stream(stream));
}

int tfcb_encode_index_f32(tfcb_encoder* h, const int32_t* index_dev, const float* y_dev,
                          const float* loc_dev, const int32_t* cdf_offset_dev, int64_t n, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not an encoder");
  return launch_encode<kModeIndex | kModeF32>(h, y_dev, index_dev, loc_dev, cdf_offset_dev, n,
                                              as_stream(stream));
}

int tfcb_encoder_check(tfcb_encoder* h, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not an encoder");
  return fetch_error(h->err, as_stream(stream), "encode");
}

int tfcb_encode_finalize(tfcb_encoder* h, void* stream, int64_t* total_bytes_host) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not an encoder");
  if (h->finalized) return fail(TFCB_INVALID_ARGUMENT, "encoder handle was already finalized");
  cudaStream_t s = as_stream(stream);
  const long long S = h->n_streams;
  // (a finalize retried after a deferred argument error reuses the buffers of the first attempt)
  if (!h->lens) TFCB_TRY(dev_alloc((void**)&h->lens, std::max<long long>(S, 1) * sizeof(long long), s));
  if (!h->offsets) TFCB_TRY(dev_alloc((void**)&h->offsets, (S + 1) * sizeof(long long), s));
  if (h->cap == 0) TFCB_TRY(ensure_capacity(h, 0, s));
  if (S > 0) {
    enc_lengths_kernel<<<(unsigned)((S + 127) / 128), 128, 0, s>>>(h->state, h->words, h->cap, S, h->lens);
    TFCB_LAUNCHED();
  }
  exclusive_scan_kernel<<<1, 1024, 0, s>>>(h->lens, S, h->offsets);
  TFCB_LAUNCHED();
  TFCB_CUDA_TRY(cudaGetLastError());
  // one host round trip for both the deferred argument errors and the total size
  long long total = 0;
  DevError err;
  if (char* scratch = static_cast<char*>(pinned_scratch())) {
    TFCB_CUDA_TRY(cudaMemcpyAsync(scratch, h->offsets + S, sizeof total, cudaMemcpyDeviceToHost, s));
    TFCB_CUDA_TRY(cudaMemcpyAsync(scratch + 64, h->err, sizeof err, cudaMemcpyDeviceToHost, s));
    TFCB_CUDA_TRY(cudaStreamSynchronize(s));
    std::memcpy(&total, scratch, sizeof total);
    std::memcpy(&err, scratch + 64, sizeof err);
  } else {
    TFCB_CUDA_TRY(cudaMemcpyAsync(&total, h->offsets + S, sizeof total, cudaMemcpyDeviceToHost, s));
    TFCB_CUDA_TRY(cudaMemcpyAsync(&err, h->err, sizeof err, cudaMemcpyDeviceToHost, s));
    TFCB_CUDA_TRY(cudaStreamSynchronize(s));
  }
  TFCB_TRY(decode_error(err, "encode"));
  h->total = total;
  TFCB_TRY(dev_alloc((void**)&h->out, (size_t)std::max<long long>(total, 1), s));
  if (S > 0) {
    enc_write_kernel<<<(unsigned)S, 32 * kWriteWarps, 0, s>>>(h->state, h->words, h->cbits, h->cap, S,
                                                             h->offsets, h->out);
    TFCB_LAUNCHED();
    TFCB_CUDA_TRY(cudaGetLastError());
  }
  // the word arena is no longer needed
  dev_free(h->words, s);
  dev_free(h->cbits, s);
  h->words = nullptr;
  h->cbits = nullptr;
  h->finalized = true;
  if (total_bytes_host) *total_bytes_host = total;
  return TFCB_OK;
}

int tfcb_encoder_output(tfcb_encoder* h, const uint8_t** bytes_dev, const int64_t** offsets_dev) {
  if (!h || !h->finalized) return fail(TFCB_INVALID_ARGUMENT, "encoder handle is not finalized");
  if (bytes_dev) *bytes_dev = h->out;
  if (offsets_dev) *offsets_dev = reinterpret_cast<const int64_t*>(h->offsets);
  return TFCB_OK;
}

int tfcb_encoder_copy_output(tfcb_encoder* h, uint8_t* bytes_host, int64_t* offsets_host, void* stream) {
  if (!h || !h->finalized) return fail(TFCB_INVALID_ARGUMENT, "encoder handle is not finalized");
  cudaStream_t s = as_stream(stream);
  if (bytes_host && h->total > 0)
    TFCB_CUDA_TRY(cudaMemcpyAsync(bytes_host, h->out, (size_t)h->total, cudaMemcpyDeviceToHost, s));
  if (offsets_host)
    TFCB_CUDA_TRY(cudaMemcpyAsync(offsets_host, h->offsets, (h->n_streams + 1) * sizeof(long long),
                                  cudaMemcpyDeviceToHost, s));
  TFCB_CUDA_TRY(cudaStreamSynchronize(s));
  return TFCB_OK;
}

void tfcb_encoder_destroy(tfcb_encoder* h) {
  if (!h) return;
  cudaStream_t s = h->home;
  lookup_cache().release(h->lut_token);
  dev_free(h->state, s);
  dev_free(h->words, s);
  dev_free(h->cbits, s);
  dev_free(h->err, s);
  dev_free(h->lens, s);
  dev_free(h->offsets, s);
  dev_free(h->out, s);
  delete h;
}

}  // extern "C"

struct tfcb_decoder {
  DeviceLookup lut;      // shallow copy of a cache entry's tables
  void* lut_token = nullptr;
  long long n_streams = 0;
  const uint8_t* bytes = nullptr;
  const long long* offsets = nullptr;
  DecState* state = nullptr;
  DevError* err = nullptr;
  uint8_t* ok = nullptr;
  cudaStream_t home = nullptr;
};

namespace {

template <int MODE>
int launch_decode(tfcb_decoder* h, const int32_t* index, void* out, const float* qoff,
                  const int32_t* coff, long long n, cudaStream_t s) {
  if (n < 0) return fail(TFCB_INVALID_ARGUMENT, "negative element count");
  if (h->n_streams == 0 || n == 0) return TFCB_OK;
  if (h->lut.n_rows == 0) return fail(TFCB_INVALID_ARGUMENT, "index=0 not in range [0, 0)");
  if (out == nullptr) return fail(TFCB_INVALID_ARGUMENT, "output is null");
  if ((MODE & kModeIndex) && index == nullptr) return fail(TFCB_INVALID_ARGUMENT, "`index` is null");
  if ((MODE & kModeF32) && coff == nullptr) return fail(TFCB_INVALID_ARGUMENT, "`cdf_offset` is null");
  DecParams P;
  P.lookup = h->lut.lookup;
  P.rows = h->lut.rows;
  P.pairs = h->lut.pairs;
  P.rows4 = h->lut.rows4;
  P.n_pairs = h->lut.n_pairs;
  P.zero_win = h->lut.zero_win;
  P.n_rows = h->lut.n_rows;
  P.lookup_len = h->lut.len;
  P.bytes = h->bytes;
  P.offsets = h->offsets;
  P.index = index;
  P.out = out;
  P.qoff = qoff;
  P.coff = coff;
  P.n = n;
  P.n_streams = h->n_streams;
  P.state = h->state;
  P.err = h->err;
  // Search keys live in shared memory whenever they fit beside the kernel's static 16 KB: up to 96 KB two CTAs
  // (streams) still share an SM; up to 200 KB one CTA per SM (cfg3's 64 NoisyNormal tables up to sigma = 256 take
  // 118 KB: from L1/L2 every slow-path search round cost a global-memory latency on the chain warp).
  const size_t smem = (size_t)((h->lut.n_pairs * 8 + 15) & ~15ll) + (size_t)h->lut.n_rows * sizeof(int4);
  if (smem <= 200 * 1024) {
    TFCB_CUDA_TRY(cudaFuncSetAttribute(decode_kernel<MODE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    decode_kernel<MODE, true><<<(unsigned)h->n_streams, 96, smem, s>>>(P);
  } else {
    decode_kernel<MODE, false><<<(unsigned)h->n_streams, 96, 0, s>>>(P);
  }
  TFCB_LAUNCHED();
  TFCB_CUDA_TRY(cudaGetLastError());
  return TFCB_OK;
}

}  // namespace

extern "C" {

int tfcb_decoder_create(const uint8_t* bytes_dev, const int64_t* offsets_dev, int64_t n_streams,
                        const int32_t* lookup_host, int64_t lookup_len, int64_t lookup_cols,
                        void* stream, tfcb_decoder** out) {
  if (!out) return fail(TFCB_INVALID_ARGUMENT, "null output handle");
  *out = nullptr;
  if (n_streams <= 0) return fail(TFCB_INVALID_ARGUMENT, "`encoded` is empty");
  if (!offsets_dev) return fail(TFCB_INVALID_ARGUMENT, "`offsets` is null");
  cudaStream_t s = as_stream(stream);
  tfcb_decoder* h = new tfcb_decoder;
  h->home = s;
  h->n_streams = n_streams;
  h->bytes = bytes_dev;
  h->offsets = reinterpret_cast<const long long*>(offsets_dev);
  int rc = lookup_cache().acquire(lookup_host, lookup_len, lookup_cols, /*for_decoder=*/true, s, &h->lut, &h->lut_token);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&h->state, n_streams * sizeof(DecState), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&h->err, sizeof(DevError), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&h->ok, n_streams, s);
  if (rc != TFCB_OK) {
    tfcb_decoder_destroy(h);
    return rc;
  }
  cudaMemsetAsync(h->err, 0, sizeof(DevError), s);
  dec_init_state_kernel<<<(unsigned)((n_streams + 255) / 256), 256, 0, s>>>(h->state, n_streams);
  TFCB_LAUNCHED();
  if (cudaGetLastError() != cudaSuccess) {
    tfcb_decoder_destroy(h);
    return fail(TFCB_CUDA_ERROR, "decoder state initialisation failed");
  }
  *out = h;
  return TFCB_OK;
}

int tfcb_decode_channel(tfcb_decoder* h, int32_t* out_dev, int64_t n, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not a decoder");
  return launch_decode<0>(h, nullptr, out_dev, nullptr, nullptr, n, as_stream(stream));
}

int tfcb_decode_index(tfcb_decoder* h, const int32_t* index_dev, int32_t* out_dev, int64_t n, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not a decoder");
  return launch_decode<kModeIndex>(h, index_dev, out_dev, nullptr, nullptr, n, as_stream(stream));
}

int tfcb_decode_channel_f32(tfcb_decoder* h, float* out_dev, const float* quant_offset_dev,
                            const int32_t* cdf_offset_dev, int64_t n, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not a decoder");
  return launch_decode<kModeF32>(h, nullptr, out_dev, quant_offset_dev, cdf_offset_dev, n, as_stream(stream));
}

int tfcb_decode_index_f32(tfcb_decoder* h, const int32_t* index_dev, float* out_dev, const float* loc_dev,
                          const int32_t* cdf_offset_dev, int64_t n, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not a decoder");
  return launch_decode<kModeIndex | kModeF32>(h, index_dev, out_dev, loc_dev, cdf_offset_dev, n,
                                              as_stream(stream));
}

int tfcb_decode_finalize(tfcb_decoder* h, uint8_t* ok_host, void* stream) {
  if (!h) return fail(TFCB_INVALID_ARGUMENT, "'handle' is not a decoder");
  cudaStream_t s = as_stream(stream);
  TFCB_TRY(fetch_error(h->err, s, "decode"));
  dec_finalize_kernel<<<(unsigned)((h->n_streams + 127) / 128), 128, 0, s>>>(h->state, h->bytes, h->offsets,
                                                                             h->n_streams, h->ok);
  TFCB_LAUNCHED();
  TFCB_CUDA_TRY(cudaGetLastError());
  if (ok_host) TFCB_CUDA_TRY(cudaMemcpyAsync(ok_host, h->ok, h->n_streams, cudaMemcpyDeviceToHost, s));
  TFCB_CUDA_TRY(cudaStreamSynchronize(s));
  return TFCB_OK;
}

void tfcb_decoder_destroy(tfcb_decoder* h) {
  if (!h) return;
  cudaStream_t s = h->home;
  lookup_cache().release(h->lut_token);
  dev_free(h->state, s);
  dev_free(h->err, s);
  dev_free(h->ok, s);
  delete h;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Legacy ops: host side
// ---------------------------------------------------------------------------------------------
namespace {

// MergeAxes of range_coding_kernels_util.cc:34-91 plus the argument checks of
// range_coding_kernels.cc:134-148,179-185.
int legacy_prepare(const int64_t* dshape, int rank, const int64_t* cshape, int crank, int precision,
                   int debug_level, LegacyDims* dims, long long* n_elems, long long* n_rows) {
  if (!(0 < precision && precision <= 16))
    return fail(TFCB_INVALID_ARGUMENT, "`precision` must be in [1, 16]: %d", precision);
  if (!(debug_level == 0 || debug_level == 1))
    return fail(TFCB_INVALID_ARGUMENT, "`debug_level` must be 0 or 1: %d", debug_level);
  if (rank < 0 || crank != rank + 1)
    return fail(TFCB_INVALID_ARGUMENT, "`cdf` should have one more axis than `data`: data rank=%d, cdf rank=%d",
                rank, crank);
  if (cshape[rank] <= 1)
    return fail(TFCB_INVALID_ARGUMENT, "The last dimension of `cdf` should be > 1: %lld",
                (long long)cshape[rank]);
  if (debug_level > 0 && cshape[rank] <= 2)
    return fail(TFCB_INVALID_ARGUMENT, "CDF size should be > 2: %lld", (long long)cshape[rank]);
  std::vector<long long> md(1, 1), mc(1, 1);
  long long n = 1, rows = 1;
  for (int j = 0; j < rank; ++j) {
    if (dshape[j] < 0) return fail(TFCB_INVALID_ARGUMENT, "negative dimension");
    if (dshape[j] != cshape[j] && cshape[j] != 1)
      return fail(TFCB_INVALID_ARGUMENT, "Cannot broadcast shape of `cdf` to the shape of `data` at axis %d (%lld vs %lld)",
                  j, (long long)cshape[j], (long long)dshape[j]);
    const bool was_b = mc.back() == 1, is_b = cshape[j] == 1;
    if (was_b == is_b || dshape[j] <= 1 || md.back() <= 1) {
      md.back() *= dshape[j];
      mc.back() *= cshape[j];
    } else {
      md.push_back(dshape[j]);
      mc.push_back(cshape[j]);
    }
    n *= dshape[j];
    rows *= cshape[j];
  }
  if (md.size() > 6)
    return fail(TFCB_INVALID_ARGUMENT, "Irregular broadcast pattern: more than 6 merged axis groups");
  dims->rank = (int)md.size();
  for (int i = 0; i < 6; ++i) {
    dims->data[i] = i < dims->rank ? md[i] : 1;
    dims->cdfd[i] = i < dims->rank ? mc[i] : 1;
  }
  dims->chip = cshape[rank];
  *n_elems = n;
  *n_rows = rows;
  return TFCB_OK;
}

}  // namespace

extern "C" {

int tfcb_range_encode(const int16_t* data_dev, const int64_t* data_shape_host, int rank,
                      const int32_t* cdf_dev, const int64_t* cdf_shape_host, int cdf_rank, int precision,
                      int debug_level, uint8_t* out_host, int64_t out_cap, int64_t* n_bytes_host,
                      void* stream) {
  cudaStream_t s = as_stream(stream);
  LegacyDims dims;
  long long n = 0, rows = 0;
  TFCB_TRY(legacy_prepare(data_shape_host, rank, cdf_shape_host, cdf_rank, precision, debug_level, &dims,
                          &n, &rows));
  const long long cap = (((n * precision + 15) / 16 + 2 + 32) + 31) & ~31ll;
  if (cap >= (1ll << 31) - 64) return fail(TFCB_INVALID_ARGUMENT, "input too large for one code stream");
  EncState* state = nullptr;
  uint16_t* words = nullptr;
  uint32_t* cbits = nullptr;
  DevError* err = nullptr;
  long long* lens = nullptr;
  uint8_t* out = nullptr;
  int rc = dev_alloc((void**)&state, sizeof(EncState), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&words, cap * sizeof(uint16_t), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&cbits, (cap >> 5) * sizeof(uint32_t), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&err, sizeof(DevError), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&lens, 3 * sizeof(long long), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&out, (size_t)(2 * cap + 8), s);
  auto cleanup = [&]() {
    dev_free(state, s);
    dev_free(words, s);
    dev_free(cbits, s);
    dev_free(err, s);
    dev_free(lens, s);
    dev_free(out, s);
  };
  if (rc != TFCB_OK) {
    cleanup();
    return rc;
  }
  cudaMemsetAsync(err, 0, sizeof(DevError), s);
  if (debug_level > 0 && rows > 0) {
    legacy_check_cdf_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, s>>>(cdf_dev, rows, dims.chip,
                                                                          precision, err);
    TFCB_LAUNCHED();
    rc = fetch_error(err, s, "legacy");
    if (rc != TFCB_OK) {
      cleanup();
      return rc;
    }
  }
  legacy_encode_kernel<<<1, 32, 0, s>>>(data_dev, n, cdf_dev, dims, precision, debug_level, state, words,
                                        cbits, cap, err);
  TFCB_LAUNCHED();
  rc = fetch_error(err, s, "legacy");
  if (rc != TFCB_OK) {
    cleanup();
    return rc;
  }
  enc_lengths_kernel<<<1, 32, 0, s>>>(state, words, cap, 1, lens);
  exclusive_scan_kernel<<<1, 32, 0, s>>>(lens, 1, lens + 1);
  enc_write_kernel<<<1, 32 * kWriteWarps, 0, s>>>(state, words, cbits, cap, 1, lens + 1, out);
  TFCB_LAUNCHED();
  TFCB_LAUNCHED();
  TFCB_LAUNCHED();
  long long total = 0;
  cudaMemcpyAsync(&total, lens, sizeof total, cudaMemcpyDeviceToHost, s);
  cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    cleanup();
    return fail(TFCB_CUDA_ERROR, "CUDA error '%s' in tfcb_range_encode", cudaGetErrorString(e));
  }
  if (n_bytes_host) *n_bytes_host = total;
  if (total > out_cap) {
    cleanup();
    return fail(TFCB_INVALID_ARGUMENT, "output buffer too small: need %lld bytes", total);
  }
  if (total > 0) cudaMemcpyAsync(out_host, out, (size_t)total, cudaMemcpyDeviceToHost, s);
  e = cudaStreamSynchronize(s);
  cleanup();
  if (e != cudaSuccess) return fail(TFCB_CUDA_ERROR, "CUDA error '%s' in tfcb_range_encode", cudaGetErrorString(e));
  return TFCB_OK;
}

int tfcb_range_decode(const uint8_t* encoded_host, int64_t n_bytes, const int64_t* shape_host, int rank,
                      const int32_t* cdf_dev, const int64_t* cdf_shape_host, int cdf_rank, int precision,
                      int debug_level, int16_t* out_dev, void* stream) {
  cudaStream_t s = as_stream(stream);
  LegacyDims dims;
  long long n = 0, rows = 0;
  TFCB_TRY(legacy_prepare(shape_host, rank, cdf_shape_host, cdf_rank, precision, debug_level, &dims, &n, &rows));
  if (n_bytes < 0) return fail(TFCB_INVALID_ARGUMENT, "negative string length");
  uint8_t* bytes = nullptr;
  DevError* err = nullptr;
  int rc = dev_alloc((void**)&bytes, (size_t)std::max<int64_t>(n_bytes, 1), s);
  if (rc == TFCB_OK) rc = dev_alloc((void**)&err, sizeof(DevError), s);
  auto cleanup = [&]() {
    dev_free(bytes, s);
    dev_free(err, s);
  };
  if (rc != TFCB_OK) {
    cleanup();
    return rc;
  }
  cudaMemsetAsync(err, 0, sizeof(DevError), s);
  if (n_bytes > 0) cudaMemcpyAsync(bytes, encoded_host, (size_t)n_bytes, cudaMemcpyHostToDevice, s);
  if (debug_level > 0 && rows > 0) {
    legacy_check_cdf_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, s>>>(cdf_dev, rows, dims.chip,
                                                                          precision, err);
    TFCB_LAUNCHED();
    rc = fetch_error(err, s, "legacy");
    if (rc != TFCB_OK) {
      cleanup();
      return rc;
    }
  }
  if (n > 0) {
    legacy_decode_kernel<<<1, 32, 0, s>>>(bytes, n_bytes, n, cdf_dev, dims, precision, out_dev);
    TFCB_LAUNCHED();
  }
  cudaError_t e = cudaStreamSynchronize(s);
  cleanup();
  if (e != cudaSuccess) return fail(TFCB_CUDA_ERROR, "CUDA error '%s' in tfcb_range_decode", cudaGetErrorString(e));
  return TFCB_OK;
}

}  // extern "C"
