// coalescer_mixed_test.cpp — the query coalescer (semadb_b200/host/coalescer.hpp) under mixed traffic:
// 32 threads send requests with random (Limit, SearchSize) and optional filters; every result must
// equal IndexVamana::Search of that request alone, the batches must be those max_batch forces (not
// one per (Limit, SearchSize) pair), and an invalid request fails alone.
// usage: coalescer_mixed_test   (needs a CUDA device)
#include <atomic>
#include <cstdio>
#include <random>
#include <thread>

#include "../../semadb_b200/host/coalescer.hpp"

using namespace semadb;
using vamana::IndexVamana;
using vamana::IndexVectorChange;

static int g_fail = 0;
#define CHECK(cond)                                                         \
  do {                                                                      \
    if (!(cond)) {                                                          \
      std::fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      ++g_fail;                                                             \
    }                                                                       \
  } while (0)

static void test_coalescer_mixed() {
  std::mt19937 rng(11);
  const unsigned dim = 16;
  models::IndexVectorVamanaParameters p;  // vamana_test.go:21-27
  p.VectorSize = dim;
  p.DistanceMetric = models::DistanceEuclidean;
  p.SearchSize = 75;
  p.DegreeBound = 64;
  p.Alpha = 1.2f;
  diskstore::MemBucket bucket;
  std::unique_ptr<IndexVamana> inv;
  if (Error e = IndexVamana::New("test", p, &bucket, &inv, 0, 5)) {
    std::fprintf(stderr, "FAIL New: %s\n", e.msg.c_str());
    ++g_fail;
    return;
  }
  std::uniform_real_distribution<float> u(0.0f, 1.0f);
  std::vector<IndexVectorChange> pts(5000);
  for (size_t i = 0; i < pts.size(); ++i) {
    pts[i].Id = uint64_t(i + 2);
    pts[i].Vector.resize(dim);
    for (unsigned d = 0; d < dim; ++d) pts[i].Vector[d] = u(rng);
  }
  if (Error e = inv->InsertUpdateDelete(pts)) {
    std::fprintf(stderr, "FAIL insert: %s\n", e.msg.c_str());
    ++g_fail;
    return;
  }
  const uint32_t B = 3000, MAXB = 16;
  std::vector<models::SearchVectorVamanaOptions> q(B);
  std::vector<std::vector<uint64_t>> filt(B);
  std::vector<bool> has_filter(B);
  for (uint32_t b = 0; b < B; ++b) {
    q[b].Vector = pts[b].Vector;
    q[b].Limit = int(std::uniform_int_distribution<int>(1, 75)(rng));
    q[b].SearchSize = int(std::uniform_int_distribution<int>(std::max(25, q[b].Limit), 75)(rng));
    has_filter[b] = b % 3 == 0;
    if (has_filter[b] && b % 30 != 0)  // every 30th: an empty filter
      for (uint64_t j = 0; j < 60 + b % 90; ++j) filt[b].push_back(pts[(b * 7 + j * 13) % pts.size()].Id);
  }
  q[1234].SearchSize = 10;           // invalid (search.go:277-306): fails alone
  filt[999].push_back(1u << 30);     // a missing point among its seeds: fails alone
  q[999].SearchSize = 75;
  std::vector<std::vector<models::SearchResult>> want(B);
  std::vector<int> want_err(B, 0);
  for (uint32_t b = 0; b < B; ++b) {
    std::vector<uint64_t> rs;
    want_err[b] = b == 1234 ? 1 : bool(inv->Search(q[b], has_filter[b] ? &filt[b] : nullptr, &rs, &want[b]));
  }
  CHECK(want_err[999] == 1 && want_err[0] == 0 && want[0].empty() && !want[3].empty());
  vamana::SearchCoalescer co(inv.get(), MAXB, std::chrono::microseconds(500));
  std::atomic<int> bad{0};
  std::vector<std::thread> th;
  for (int t = 0; t < 32; ++t)
    th.emplace_back([&, t] {
      for (uint32_t b = t; b < B; b += 32) {
        std::vector<uint64_t> rs;
        std::vector<models::SearchResult> res;
        Error e = co.Search(q[b], has_filter[b] ? &filt[b] : nullptr, &rs, &res);
        if (bool(e) != bool(want_err[b])) {
          std::fprintf(stderr, "request %u: error %d, want %d (%s)\n", b, int(bool(e)), want_err[b], e.msg.c_str());
          ++bad;
          continue;
        }
        if (e) continue;
        if (res.size() != want[b].size()) { ++bad; continue; }
        for (size_t j = 0; j < res.size(); ++j)
          if (res[j].NodeId != want[b][j].NodeId || res[j].Distance != want[b][j].Distance) ++bad;
      }
    });
  for (auto& x : th) x.join();
  CHECK(bad.load() == 0);
  CHECK(co.queries() == B - 1);  // the invalid request never reached the queue
  // 32 callers, at most MAXB per batch: a batch takes whatever waits, so about B / MAXB batches;
  // batching by (Limit, SearchSize) would need several per round
  const uint64_t forced = (B + MAXB - 1) / MAXB;
  std::fprintf(stderr, "coalescer mixed: %llu queries in %llu batches (max_batch forces %llu)\n",
               (unsigned long long)co.queries(), (unsigned long long)co.batches(), (unsigned long long)forced);
  CHECK(co.batches() <= forced + forced / 4 + 8);
}

int main() {
  if (sdb_device_count() == 0) {
    std::fprintf(stderr, "no CUDA device: the GPU index has no CPU fallback\n");
    return 2;
  }
  test_coalescer_mixed();
  if (g_fail) {
    std::fprintf(stderr, "%d check(s) failed\n", g_fail);
    return 1;
  }
  std::printf("coalescer_mixed_test: ok\n");
  return 0;
}
