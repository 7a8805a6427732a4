// scorecut.hpp -- host policy of an iteration (a12): the score / length regression of find_fsdb_score_cut
// (fsdb.c:269-383) and the per-read test of cull_maln_from_fsdb (mia.c:418-479).  Host C++ only.
//
// The reference forms two sums in double precision, one read after the other in FSDB order:
//     ssxy += (len - xbar) * (score - ybar);      ssxx += (len - xbar) * (len - xbar);
// Every addition rounds, so the result depends on the order and the obvious parallel sum is not bit-identical.
// chained_sum() evaluates exactly that left-to-right chain, but block-wise: while the running sum S stays inside
// one binade [2^e, 2^(e+1)) it is an integer multiple N of ulp = 2^(e-52), and fl(S + a) = ulp * (N + rint(a / ulp))
// unless a / ulp is an exact tie.  A block of addends therefore moves S by ulp * sum(rint(a_i / ulp)) -- an integer
// sum that any number of threads can take in any order -- provided no partial sum leaves the binade, which
// N0 +- sum(|rint(a_i / ulp)|) bounds.  Blocks that fail the test (a binade crossing, a tie, the first few reads)
// are added one read at a time exactly as the reference does.  No test checks chained_sum() on its own:
// tests/test_oracle_vs_ref.py (test_score_cut_matches_reference_regression) compares the whole cut, block path
// included above 2,048 reads, with the oracle's plain chain on batches of up to 4,000 reads, and the session tests
// compare the resulting dropped flags with the reference's.
#pragma once
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

namespace miagpu {

// A team of host threads that runs one function on every member; the caller is member 0.
class HostTeam {
 public:
  explicit HostTeam(int threads) : n_(std::max(1, threads)) {
    for (int t = 1; t < n_; t++) workers_.emplace_back([this, t] { loop(t); });
  }
  ~HostTeam() {
    { std::lock_guard<std::mutex> g(m_); stop_ = true; gen_++; }
    cv_.notify_all();
    for (auto& w : workers_) w.join();
  }
  int size() const { return n_; }
  void run(const std::function<void(int)>& f) {
    if (n_ == 1) { f(0); return; }
    { std::lock_guard<std::mutex> g(m_); job_ = &f; pending_ = n_ - 1; gen_++; }
    cv_.notify_all();
    f(0);
    std::unique_lock<std::mutex> g(m_);
    done_.wait(g, [this] { return pending_ == 0; });
    job_ = nullptr;
  }
  // slices [lo, hi) of [0, n) per member
  template <typename F>
  void chunks(int64_t n, F f) {
    run([&](int t) { f(t, n * t / n_, n * (t + 1) / n_); });
  }

 private:
  void loop(int t) {
    uint64_t seen = 0;
    for (;;) {
      const std::function<void(int)>* job;
      {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [&] { return gen_ != seen; });
        seen = gen_;
        if (stop_) return;
        job = job_;
      }
      if (job) (*job)(t);
      { std::lock_guard<std::mutex> g(m_); pending_--; }
      done_.notify_one();
    }
  }
  int n_;
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  const std::function<void(int)>* job_ = nullptr;
  int pending_ = 0;
  uint64_t gen_ = 0;
  bool stop_ = false;
};

// 512: a block the stitch cannot prove costs 512 dependent additions on the host (about 25 such blocks per chain and million
// reads: the first one and the binade crossings); smaller blocks would only add records
constexpr int64_t CHAIN_BLOCK = 512;

// What phases 1 and 2 know about one block of CHAIN_BLOCK consecutive addends: the binade e the running sum is
// predicted to be in when the block starts, T = sum(rint(a_i / ulp_e)), A = sum(|rint(a_i / ulp_e)|), and ok =
// every quotient was far from a tie and all partial integer sums were exact.  The host team below fills these,
// and so do the device kernels of scorecut.cuh (same arithmetic, IEEE double, no contraction).
struct ChainBlock { double approx, T, A; int e; bool ok; };

// phase 3: stitch the blocks in order; whatever cannot be proven goes read by read, exactly as the reference adds.
// serial(b, S) returns S after the addends of block b have been added one at a time.
template <typename Serial>
double chain_stitch_blocks(const ChainBlock* blk, int64_t nb, const Serial& serial, int64_t* n_serial = nullptr) {
  double S = 0;
  int64_t count = 0;
  int e_cached = INT32_MIN;                           // the scale factors change only when the running sum changes binade
  double inv = 0, ulp = 0, lo = 0, hi = 0;            // lo <= S < hi: S is in binade e_cached
  for (int64_t b = 0; b < nb; b++) {
    const ChainBlock& B = blk[b];
    if (B.ok && S > 0) {
      if (!(S >= lo && S < hi)) {
        e_cached = std::ilogb(S);
        inv = std::ldexp(1.0, 52 - e_cached); ulp = std::ldexp(1.0, e_cached - 52);
        lo = std::ldexp(1.0, e_cached); hi = std::ldexp(1.0, e_cached + 1);
      }
      if (e_cached == B.e) {
        const double N0 = S * inv;                    // integer in [2^52, 2^53)
        if (N0 - B.A >= 4503599627370497.0 && N0 + B.A <= 9007199254740990.0) {
          S = (N0 + B.T) * ulp;
          continue;
        }
      }
    }
    S = serial(b, S);
    count++;
  }
  if (n_serial) *n_serial = count;
  return S;
}
template <typename Addend>
double chain_stitch(int64_t n, const Addend& a, const ChainBlock* blk, int64_t nb, int64_t* n_serial = nullptr) {
  return chain_stitch_blocks(blk, nb, [&](int64_t b, double S) {
    const int64_t i1 = std::min(n, (b + 1) * CHAIN_BLOCK);
    for (int64_t i = b * CHAIN_BLOCK; i < i1; i++) S += a(i);
    return S;
  }, n_serial);
}

// (((0 + a(0)) + a(1)) + ... + a(n-1)) with a rounding after every addition, bit-identical to the plain loop.
template <typename Addend>
double chained_sum(int64_t n, const Addend& a, HostTeam& team) {
  const int64_t nb = (n + CHAIN_BLOCK - 1) / CHAIN_BLOCK;
  if (nb <= 4) {
    double s = 0;
    for (int64_t i = 0; i < n; i++) s += a(i);
    return s;
  }
  std::vector<ChainBlock> blk(nb);
  // phase 1: plain block sums -> approximate running sum at every block start (predicts the binade)
  team.chunks(nb, [&](int, int64_t b0, int64_t b1) {
    for (int64_t b = b0; b < b1; b++) {
      const int64_t i1 = std::min(n, (b + 1) * CHAIN_BLOCK);
      double s0 = 0, s1 = 0;
      int64_t i = b * CHAIN_BLOCK;
      for (; i + 1 < i1; i += 2) { s0 += a(i); s1 += a(i + 1); }
      if (i < i1) s0 += a(i);
      blk[b].approx = s0 + s1;
    }
  });
  double run = 0;
  for (int64_t b = 0; b < nb; b++) { const double p = blk[b].approx; blk[b].approx = run; run += p; }
  // phase 2: integer increments of every block in the predicted binade
  constexpr double MAGIC = 6755399441055744.0;       // 1.5 * 2^52: (x + MAGIC) - MAGIC = x rounded to nearest-even for |x| < 2^51
  team.chunks(nb, [&](int, int64_t b0, int64_t b1) {
    for (int64_t b = b0; b < b1; b++) {
      ChainBlock& B = blk[b];
      B.ok = false;
      const double s = B.approx;
      if (!(s > 0) || !std::isfinite(s)) continue;
      int e2 = 0;
      const double f = std::frexp(s, &e2);            // s = f * 2^e2, f in [0.5, 1)
      if (f < 0.5 + 1e-6 || f > 1 - 1e-6) continue;   // too close to a binade boundary to predict
      B.e = e2 - 1;
      if (B.e < -900 || B.e > 900) continue;
      const double inv = std::ldexp(1.0, 52 - B.e);   // 1 / ulp
      const int64_t i0 = b * CHAIN_BLOCK, i1 = std::min(n, (b + 1) * CHAIN_BLOCK);
      double T0 = 0, T1 = 0, A0 = 0, A1 = 0;
      bool bad = false;
      int64_t i = i0;
      for (; i + 1 < i1; i += 2) {
        const double x0 = a(i) * inv, x1 = a(i + 1) * inv;
        const double m0 = (x0 + MAGIC) - MAGIC, m1 = (x1 + MAGIC) - MAGIC;
        bad |= !(std::fabs(x0) < 1125899906842624.0) | !(std::fabs(x1) < 1125899906842624.0);   // 2^50
        bad |= (std::fabs(x0 - m0) == 0.5) | (std::fabs(x1 - m1) == 0.5);                        // exact ties round by parity
        T0 += m0; T1 += m1; A0 += std::fabs(m0); A1 += std::fabs(m1);
      }
      if (i < i1) {
        const double x0 = a(i) * inv;
        const double m0 = (x0 + MAGIC) - MAGIC;
        bad |= !(std::fabs(x0) < 1125899906842624.0) | (std::fabs(x0 - m0) == 0.5);
        T0 += m0; A0 += std::fabs(m0);
      }
      B.T = T0 + T1;
      B.A = A0 + A1;
      B.ok = !bad && B.A < 4503599627370496.0;        // 2^52: all partial integer sums were exact
    }
  });
  return chain_stitch(n, a, blk.data(), nb);
}

}  // namespace miagpu
