// coalescer.hpp — turns the reference's call pattern (one goroutine per request, each calling
// IndexVamana.Search with ONE vector under a read lock: shard/index/search.go:67-85,
// shard/cache/manager.go:151-182) into the batches the GPU kernels need (SURVEY.md §8f-1).
// Callers block in Search(); a single batcher thread collects requests until `max_batch` are
// waiting or the oldest has waited `window`, runs one sdb_search_batch_requests for all of them —
// each with its own limit, searchSize (models/search.go:268-314) and optional filter bitmap, like
// shard/index/search.go:59-85 — and hands every caller its own slice of the result.
#pragma once
#include <chrono>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

#include "gpuvamana.hpp"

namespace semadb {
namespace vamana {

class SearchCoalescer {
 public:
  SearchCoalescer(IndexVamana* index, uint32_t max_batch = 1024,
                  std::chrono::microseconds window = std::chrono::microseconds(200))
      : ix_(index), max_batch_(max_batch ? max_batch : 1), window_(window), worker_([this] { Run(); }) {}
  ~SearchCoalescer() {
    {
      std::lock_guard<std::mutex> g(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    worker_.join();
  }

  // Same contract as IndexVamana::Search (filter: nullptr = none, empty = matches nothing);
  // thread-safe, blocking.
  Error Search(const models::SearchVectorVamanaOptions& query, std::vector<uint64_t>* result_set,
               std::vector<models::SearchResult>* results) {
    return Search(query, nullptr, result_set, results);
  }
  Error Search(const models::SearchVectorVamanaOptions& query, const std::vector<uint64_t>* filter,
               std::vector<uint64_t>* result_set, std::vector<models::SearchResult>* results) {
    if (query.Vector.size() != ix_->Parameters().VectorSize)
      return Error("could not perform graph search: query vector length mismatch");
    // an invalid request fails alone, before it can fail the batch it would have joined
    if (Error e = query.Validate()) return e;
    Request r;
    r.q = &query;
    r.filter = filter;
    {
      std::unique_lock<std::mutex> g(mu_);
      queue_.push_back(&r);
      cv_.notify_all();
      r.cv.wait(g, [&] { return r.done; });
    }
    if (r.err) return r.err;
    const float weight = query.Weight ? *query.Weight : 1.0f;
    results->clear();
    result_set->clear();
    for (uint32_t i = 0; i < r.count; ++i) {
      models::SearchResult sr;
      sr.NodeId = r.ids[i];
      sr.Distance = r.dists[i];
      sr.HybridScore = -1.0f * r.dists[i] * weight;
      results->push_back(sr);
      result_set->push_back(r.ids[i]);
    }
    std::sort(result_set->begin(), result_set->end());
    return Ok();
  }

  uint64_t batches() const { return batches_; }
  uint64_t queries() const { return queries_; }

 private:
  struct Request {
    const models::SearchVectorVamanaOptions* q = nullptr;
    const std::vector<uint64_t>* filter = nullptr;
    std::vector<uint64_t> ids;
    std::vector<float> dists;
    uint32_t count = 0;
    Error err;
    bool done = false;
    std::condition_variable cv;
  };

  void Run() {
    const uint32_t dim = ix_->Parameters().VectorSize;
    std::vector<float> qbuf;
    std::vector<uint64_t> ids;
    std::vector<float> dists;
    std::vector<uint32_t> counts, limits, sizes;
    std::unique_lock<std::mutex> g(mu_);
    for (;;) {
      cv_.wait(g, [&] { return stop_ || !queue_.empty(); });
      if (queue_.empty()) {
        if (stop_) return;
        continue;
      }
      // let the batch fill up, but never hold the oldest request longer than `window`
      const auto deadline = std::chrono::steady_clock::now() + window_;
      cv_.wait_until(g, deadline, [&] { return stop_ || queue_.size() >= max_batch_; });
      // take the waiting requests in arrival order, whatever their (limit, searchSize)
      std::vector<Request*> batch;
      while (!queue_.empty() && batch.size() < max_batch_) {
        batch.push_back(queue_.front());
        queue_.pop_front();
      }
      g.unlock();
      const uint32_t B = uint32_t(batch.size());
      qbuf.resize(size_t(B) * dim);
      limits.resize(B);
      sizes.resize(B);
      uint32_t kk = 1;  // row stride: the largest limit of the batch
      for (uint32_t b = 0; b < B; ++b) {
        std::copy(batch[b]->q->Vector.begin(), batch[b]->q->Vector.end(), qbuf.begin() + size_t(b) * dim);
        limits[b] = uint32_t(batch[b]->q->Limit);
        sizes[b] = uint32_t(batch[b]->q->SearchSize);
        kk = std::max(kk, limits[b]);
      }
      ids.assign(size_t(B) * kk, 0);
      dists.assign(size_t(B) * kk, 0.0f);
      counts.assign(B, 0);
      std::vector<const std::vector<uint64_t>*> filters(B, nullptr);
      bool any_filter = false;
      for (uint32_t b = 0; b < B; ++b) {
        filters[b] = batch[b]->filter;
        any_filter |= batch[b]->filter != nullptr;
      }
      if (!any_filter) filters.clear();
      std::vector<Error> errs(B);
      Error err = ix_->SearchBatchRequests(qbuf.data(), B, limits.data(), sizes.data(), filters, kk, ids.data(), dists.data(),
                                           counts.data());
      if (err && any_filter && B > 1) {
        // a request whose filter names a missing point fails alone in the reference (search.go:45-48):
        // re-run the batch request by request so only the offender gets the error
        for (uint32_t b = 0; b < B; ++b) {
          std::vector<const std::vector<uint64_t>*> one(1, filters[b]);
          errs[b] = ix_->SearchBatchRequests(qbuf.data() + size_t(b) * dim, 1, &limits[b], &sizes[b], one, limits[b],
                                             ids.data() + size_t(b) * kk, dists.data() + size_t(b) * kk, counts.data() + b);
        }
      } else {
        for (uint32_t b = 0; b < B; ++b) errs[b] = err;
      }
      g.lock();
      ++batches_;
      queries_ += B;
      for (uint32_t b = 0; b < B; ++b) {
        Request* r = batch[b];
        r->err = errs[b];
        if (!errs[b]) {
          r->count = counts[b];
          r->ids.assign(ids.begin() + size_t(b) * kk, ids.begin() + size_t(b) * kk + counts[b]);
          r->dists.assign(dists.begin() + size_t(b) * kk, dists.begin() + size_t(b) * kk + counts[b]);
        }
        r->done = true;
        r->cv.notify_one();
      }
    }
  }

  IndexVamana* ix_;
  size_t max_batch_;
  std::chrono::microseconds window_;
  std::mutex mu_;
  std::condition_variable cv_;
  std::deque<Request*> queue_;
  bool stop_ = false;
  uint64_t batches_ = 0, queries_ = 0;
  std::thread worker_;
};

}  // namespace vamana
}  // namespace semadb
