// gpuvamana.hpp — C++ host side of the GPU Vamana index: the same surface the reference's Go
// type exposes to its callers (shard/index/vamana/vamana.go), over the C ABI in
// include/semadb_b200.h. The reference host language is Go; no Go toolchain exists in the build
// image, so this is the compiled-language mirror (the cgo stub is in INTEGRATION.md).
//
//   NewIndexVamana(name, params, bucket)   vamana.go:54-81   hydrate from the bucket keys
//   SizeInMemory()                         vamana.go:83-85   (cache.Cachable)
//   UpdateBucket(bucket)                   vamana.go:87-91
//   InsertUpdateDelete(changes)            vamana.go:127-263 classify, insert, removeInboundEdges,
//                                                            delete, re-insert, Fit, flush
//   Search(options, filter)                vamana.go:278-310
//   SearchBatch(...)                       new: one C call per batch (never per distance)
//
// Persistence is unchanged (SURVEY.md §5): n<id>v LE f32 vector, n<id>q codes / bit words,
// n<id>e LE u64 edges, _vamanaMaxNodeId, _binaryQuantizerThreshold,
// _productQuantizerCentroidDists, _productQuantizerFlatCentroids (node.go:96-135,
// plain.go:125-147, binary.go:236-320, product.go:307-393, vamana.go:265-276).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <limits>
#include <memory>
#include <mutex>
#include <random>
#include <string>
#include <vector>

#include "../../include/semadb_b200.h"
#include "conversion.hpp"
#include "diskstore.hpp"
#include "models.hpp"

namespace semadb {
namespace vamana {

constexpr uint64_t STARTID = 1;                                  // vamana.go:28
constexpr const char* MAXNODEIDKEY = "_vamanaMaxNodeId";         // vamana.go:31
constexpr const char* binaryQuantizerThresholdKey = "_binaryQuantizerThreshold";            // binary.go:16
constexpr const char* productQuantizerCentroidDistsKey = "_productQuantizerCentroidDists";  // product.go:17
constexpr const char* productQuantizerFlatCentroidsKey = "_productQuantizerFlatCentroids";  // product.go:18

struct IndexVectorChange {  // vamana.go:122-125: empty Vector with IsDelete = nil vector
  uint64_t Id = 0;
  std::vector<float> Vector;
  bool IsDelete() const { return Vector.empty(); }
};

inline Error CErr(int rc, const char* what) {
  if (rc == SDB_OK) return Ok();
  const char* m = sdb_last_error();
  return Error(std::string(what) + ": " + (m ? m : "unknown error"));
}

class IndexVamana {
 public:
  // NewIndexVamana (vamana.go:54-81). start_seed draws node 1's vector when the bucket has
  // none (setupStartNode, vamana.go:93-120, is unseeded in the reference).
  static Error New(const std::string& name, const models::IndexVectorVamanaParameters& params, diskstore::Bucket* bucket,
                   std::unique_ptr<IndexVamana>* out, int device = 0, uint64_t start_seed = std::random_device{}()) {
    if (Error e = params.Validate()) return e;
    std::unique_ptr<IndexVamana> ix(new IndexVamana(name, params, bucket));
    sdb_params p{};
    if (Error e = ix->FillParams(device, &p)) return e.Wrap("could not create vector store");
    if (Error e = CErr(sdb_index_create(&p, &ix->h_), "could not create vector store")) return e;
    ix->rng_.seed(start_seed);
    if (Error e = ix->Hydrate()) return e;
    if (Error e = ix->SetupStartNode()) return e.Wrap("could not setup start node");
    *out = std::move(ix);
    return Ok();
  }
  ~IndexVamana() {
    if (h_) sdb_index_destroy(h_);
  }
  IndexVamana(const IndexVamana&) = delete;
  IndexVamana& operator=(const IndexVamana&) = delete;

  int64_t SizeInMemory() const { return sdb_index_size_bytes(h_); }  // vamana.go:83-85
  void UpdateBucket(diskstore::Bucket* bucket) { bucket_ = bucket; }   // vamana.go:87-91
  uint64_t MaxNodeId() const { return max_node_id_; }
  sdb_index* Handle() const { return h_; }
  const models::IndexVectorVamanaParameters& Parameters() const { return params_; }

  // InsertUpdateDelete (vamana.go:127-263). The Go signature is a channel in and an error
  // channel out; here the drained queue is a vector and the first error is returned.
  Error InsertUpdateDelete(const std::vector<IndexVectorChange>& changes) {
    std::lock_guard<std::mutex> g(write_mu_);  // one writer at a time (manager.go:191-205)
    const uint32_t dim = params_.VectorSize;
    std::vector<uint64_t> ids;
    std::vector<float> vecs;
    std::vector<uint8_t> has;
    ids.reserve(changes.size());
    vecs.resize(changes.size() * size_t(dim), 0.0f);
    has.reserve(changes.size());
    for (size_t i = 0; i < changes.size(); ++i) {
      const IndexVectorChange& c = changes[i];
      if (c.Id == STARTID)
        return Error("could not distribute or insert points: cannot modify point with start id: " + std::to_string(STARTID));
      if (c.Id == 0) return Error("could not distribute or insert points: invalid point id: 0");
      if (!c.IsDelete() && c.Vector.size() != dim)
        return Error("could not set point: vector length mismatch, expected " + std::to_string(dim));
      ids.push_back(c.Id);
      has.push_back(c.IsDelete() ? 0 : 1);
      if (!c.IsDelete()) std::copy(c.Vector.begin(), c.Vector.end(), vecs.begin() + i * size_t(dim));
    }
    if (!ids.empty()) {
      if (Error e = CErr(sdb_insert_update_delete(h_, ids.size(), ids.data(), vecs.data(), has.data()),
                         "could not distribute or insert points"))
        return e;
      for (size_t i = 0; i < ids.size(); ++i) {
        const bool existed = Alive(ids[i]);
        if (has[i]) {
          SetAlive(ids[i], true);
          dirty_vec_.push_back(ids[i]);
          if (ids[i] > max_node_id_) max_node_id_ = ids[i];  // vamana.go:166-168
        } else if (existed) {
          SetAlive(ids[i], false);
          deleted_.push_back(ids[i]);
        }
      }
    }
    // vecStore.Fit() (vamana.go:258): the first k-means centre is drawn at random (kmeans.go:61)
    int32_t fitted = 0;
    const uint64_t cnt = sdb_index_count(h_);
    const uint64_t first = cnt ? std::uniform_int_distribution<uint64_t>(0, cnt - 1)(rng_) : 0;
    if (Error e = CErr(sdb_index_fit(h_, first, &fitted), "could not fit vector store")) return e;
    if (fitted) {
      quant_fitted_ = true;
      all_vec_dirty_ = true;  // every point was re-encoded (binary.go:176-180, product.go:216-218)
    }
    return Flush();
  }

  // Search (vamana.go:278-310). filter: node ids of the roaring bitmap, any order.
  Error Search(const models::SearchVectorVamanaOptions& query, const std::vector<uint64_t>* filter,
               std::vector<uint64_t>* result_set, std::vector<models::SearchResult>* results) {
    if (query.Vector.size() != params_.VectorSize)
      return Error("could not perform graph search: query vector length mismatch");
    std::vector<uint64_t> ids(query.Limit > 0 ? query.Limit : 1);
    std::vector<float> d(ids.size());
    uint32_t cnt = 0;
    // A non-nil filter — empty included: it then seeds nothing and nothing can be returned
    // (search.go:33-51,93-95) — goes through the per-request entry point, which does not read
    // "filtered" off the data pointer (an empty std::vector's data() may be null).
    std::vector<uint64_t> f;
    int rc;
    if (filter) {
      f = *filter;
      std::sort(f.begin(), f.end());
      f.erase(std::unique(f.begin(), f.end()), f.end());
      const uint64_t off[2] = {0, f.size()};
      rc = sdb_search_batch_filters(h_, 1, query.Vector.data(), uint32_t(query.Limit), uint32_t(query.SearchSize), 1,
                                    f.data(), off, nullptr, ids.data(), d.data(), &cnt);
    } else {
      rc = sdb_search_batch(h_, 1, query.Vector.data(), uint32_t(query.Limit), uint32_t(query.SearchSize), nullptr, 0,
                            ids.data(), d.data(), &cnt);
    }
    if (Error e = CErr(rc, "could not perform graph search")) return e;
    const float weight = query.Weight ? *query.Weight : 1.0f;
    results->clear();
    result_set->clear();
    for (uint32_t i = 0; i < cnt; ++i) {
      models::SearchResult sr;
      sr.NodeId = ids[i];
      sr.Distance = d[i];
      sr.HybridScore = -1.0f * d[i] * weight;  // vamana.go:303
      results->push_back(sr);
      result_set->push_back(ids[i]);
    }
    std::sort(result_set->begin(), result_set->end());
    return Ok();
  }

  // The batched entry point the reference lacks: B queries, one kernel launch.
  Error SearchBatch(const float* queries, uint32_t B, uint32_t k, uint32_t search_size, uint64_t* out_ids,
                    float* out_dists, uint32_t* out_counts) {
    return CErr(sdb_search_batch(h_, B, queries, k, search_size, nullptr, 0, out_ids, out_dists, out_counts),
                "could not perform graph search");
  }

  // B requests, each with its own optional filter (nullptr = none; an empty vector is a filter
  // that matches nothing), one kernel launch per kind: what shard/index/search.go:59-85 does
  // request by request.
  Error SearchBatchFilters(const float* queries, uint32_t B, uint32_t k, uint32_t search_size,
                           const std::vector<const std::vector<uint64_t>*>& filters, uint64_t* out_ids, float* out_dists,
                           uint32_t* out_counts) {
    if (filters.size() != B) return Error("could not perform graph search: one filter slot per request expected");
    std::vector<uint64_t> flat, off(1, 0);
    std::vector<int32_t> qf(B, -1);
    std::vector<uint64_t> f;
    for (uint32_t b = 0; b < B; ++b) {
      if (!filters[b]) continue;
      f = *filters[b];
      std::sort(f.begin(), f.end());
      f.erase(std::unique(f.begin(), f.end()), f.end());
      qf[b] = int32_t(off.size() - 1);
      flat.insert(flat.end(), f.begin(), f.end());
      off.push_back(flat.size());
    }
    const uint32_t nf = uint32_t(off.size() - 1);
    return CErr(sdb_search_batch_filters(h_, B, queries, k, search_size, nf, flat.data(), off.data(), qf.data(), out_ids,
                                         out_dists, out_counts),
                "could not perform graph search");
  }

  // B requests, each with its own limit and searchSize (models/search.go:268-314) and optional filter
  // (filters empty = nobody is filtered; else one slot per request as in SearchBatchFilters), in one
  // call: outputs B x k_stride, row b holds out_counts[b] <= limits[b] results and equals the request
  // served alone.
  Error SearchBatchRequests(const float* queries, uint32_t B, const uint32_t* limits, const uint32_t* search_sizes,
                            const std::vector<const std::vector<uint64_t>*>& filters, uint32_t k_stride, uint64_t* out_ids,
                            float* out_dists, uint32_t* out_counts) {
    if (!filters.empty() && filters.size() != B)
      return Error("could not perform graph search: one filter slot per request expected");
    std::vector<uint64_t> flat, off(1, 0), f;
    std::vector<sdb_request> req(B);
    for (uint32_t b = 0; b < B; ++b) {
      req[b] = sdb_request{limits[b], search_sizes[b], 0, -1};
      if (filters.empty() || !filters[b]) continue;
      f = *filters[b];
      std::sort(f.begin(), f.end());
      f.erase(std::unique(f.begin(), f.end()), f.end());
      req[b].filter = int32_t(off.size() - 1);
      flat.insert(flat.end(), f.begin(), f.end());
      off.push_back(flat.size());
    }
    const uint32_t nf = uint32_t(off.size() - 1);
    return CErr(sdb_search_batch_requests(h_, B, queries, req.data(), nf, flat.data(), off.data(), k_stride, out_ids,
                                          out_dists, out_counts),
                "could not perform graph search");
  }

  // flush (vamana.go:265-276): vecStore.Flush, nodeStore.Flush, MAXNODEIDKEY.
  Error Flush() {
    if (bucket_ == nullptr || bucket_->IsReadOnly()) return Ok();
    if (Error e = FlushVectors()) return e.Wrap("could not flush vector store");
    if (Error e = FlushEdges()) return e.Wrap("could not flush node store");
    if (Error e = bucket_->Put(MAXNODEIDKEY, conversion::Uint64ToBytes(max_node_id_)))
      return e.Wrap("could not set max node id");
    return Ok();
  }

 private:
  IndexVamana(std::string name, models::IndexVectorVamanaParameters params, diskstore::Bucket* bucket)
      : name_(std::move(name)), params_(std::move(params)), bucket_(bucket) {}

  static int MetricCode(const std::string& m) {
    if (m == models::DistanceEuclidean) return SDB_METRIC_EUCLIDEAN;
    if (m == models::DistanceDot) return SDB_METRIC_DOT;
    if (m == models::DistanceCosine) return SDB_METRIC_COSINE;
    if (m == models::DistanceHamming) return SDB_METRIC_HAMMING;
    if (m == models::DistanceJaccard) return SDB_METRIC_JACCARD;
    if (m == models::DistanceHaversine) return SDB_METRIC_HAVERSINE;
    return -1;
  }

  // vectorstore.New (vectorstore.go:47-96)
  Error FillParams(int device, sdb_params* p) {
    p->dim = params_.VectorSize;
    p->metric = MetricCode(params_.DistanceMetric);
    p->search_size = uint32_t(params_.SearchSize);
    p->degree_bound = uint32_t(params_.DegreeBound);
    p->alpha = params_.Alpha;
    p->quantizer = SDB_QUANT_NONE;
    p->bq_threshold = std::numeric_limits<float>::quiet_NaN();
    p->bq_metric = SDB_METRIC_HAMMING;
    p->device = device;
    if (params_.Quantizer_ && params_.Quantizer_->Type != models::QuantizerNone) {
      const models::Quantizer& q = *params_.Quantizer_;
      if (q.Type == models::QuantizerBinary) {
        if (!q.Binary) return Error("binary quantizer parameters are nil");  // vectorstore.go:83
        p->quantizer = SDB_QUANT_BINARY;
        if (q.Binary->Threshold) p->bq_threshold = *q.Binary->Threshold;
        p->bq_metric = MetricCode(q.Binary->DistanceMetric);
        p->bq_trigger = uint32_t(q.Binary->TriggerThreshold);
      } else if (q.Type == models::QuantizerProduct) {
        if (!q.Product) return Error("product quantizer parameters are nil");  // vectorstore.go:88
        p->quantizer = SDB_QUANT_PRODUCT;
        p->pq_subvectors = uint32_t(q.Product->NumSubVectors);
        p->pq_centroids = uint32_t(q.Product->NumCentroids);
        p->pq_trigger = uint32_t(q.Product->TriggerThreshold);
      } else {
        return Error("unknown quantizer type " + q.Type);
      }
    }
    const bool bit_metric = params_.DistanceMetric == models::DistanceHamming || params_.DistanceMetric == models::DistanceJaccard;
    quant_kind_ = bit_metric ? SDB_QUANT_BINARY : p->quantizer;  // vectorstore.go:56-66
    quant_fitted_ = bit_metric || (p->quantizer == SDB_QUANT_BINARY && !std::isnan(p->bq_threshold));
    pqM_ = p->pq_subvectors;
    pqK_ = p->pq_centroids;
    return Ok();
  }

  bool Alive(uint64_t id) const { return id < alive_.size() && alive_[id]; }
  void SetAlive(uint64_t id, bool v) {
    if (id >= alive_.size()) alive_.resize(std::max<size_t>(id + 1, alive_.size() * 2), 0);
    alive_[id] = v ? 1 : 0;
  }
  size_t CodeWidth() const {
    return quant_kind_ == SDB_QUANT_PRODUCT ? pqM_ : 8 * ((size_t(params_.VectorSize) + 63) / 64);
  }

  // Read every n<id>{v,q,e} key plus the quantizer side keys into the device index.
  Error Hydrate() {
    if (bucket_ == nullptr) return Ok();
    std::string val;
    const uint32_t dim = params_.VectorSize;
    if (quant_kind_ == SDB_QUANT_BINARY && bucket_->Get(binaryQuantizerThresholdKey, &val)) {  // binary.go:55-61
      std::vector<float> thr = conversion::BytesToFloat32(val);
      if (thr.size() != dim) return Error("binary quantizer threshold has the wrong length");
      if (Error e = CErr(sdb_index_set_bq_threshold(h_, thr.data()), "could not load binary quantizer threshold")) return e;
      quant_fitted_ = true;
    }
    if (quant_kind_ == SDB_QUANT_PRODUCT && bucket_->Get(productQuantizerFlatCentroidsKey, &val)) {  // product.go:81-95
      std::vector<float> fc = conversion::BytesToFloat32(val);
      std::string cdv;
      if (!bucket_->Get(productQuantizerCentroidDistsKey, &cdv)) return Error("product quantizer centroid distances are missing");
      std::vector<float> cd = conversion::BytesToFloat32(cdv);
      if (fc.size() != size_t(pqM_) * pqK_ * (dim / pqM_) || cd.size() != size_t(pqM_) * pqK_ * pqK_)
        return Error("product quantizer tables have the wrong size");
      if (Error e = CErr(sdb_index_set_pq(h_, fc.data(), cd.data()), "could not load product quantizer")) return e;
      quant_fitted_ = true;
    }
    if (bucket_->Get(MAXNODEIDKEY, &val)) max_node_id_ = conversion::BytesToUint64(val);  // vamana.go:74-76
    std::vector<uint64_t> vid, qid, eid;
    std::vector<float> vdata;
    std::vector<uint8_t> qdata;
    std::vector<std::vector<uint64_t>> elists;
    const size_t cw = CodeWidth();
    Error e = bucket_->PrefixScan("n", [&](const std::string& k, const std::string& v) -> Error {
      uint64_t id = 0;
      if (conversion::NodeIdFromKey(k, 'v', &id)) {
        if (v.size() != size_t(dim) * 4) return Error("stored vector has the wrong length for node " + std::to_string(id));
        std::vector<float> f = conversion::BytesToFloat32(v);
        vid.push_back(id);
        vdata.insert(vdata.end(), f.begin(), f.end());
      } else if (conversion::NodeIdFromKey(k, 'q', &id)) {
        if (v.size() != cw) return Error("stored code has the wrong length for node " + std::to_string(id));
        qid.push_back(id);
        qdata.insert(qdata.end(), v.begin(), v.end());
      } else if (conversion::NodeIdFromKey(k, 'e', &id)) {
        eid.push_back(id);
        elists.push_back(conversion::BytesToEdgeList(v));
      }
      return Ok();
    });
    if (e) return e.Wrap("could not read index from bucket");
    if (!qid.empty()) {
      if (!quant_fitted_) return Error("quantized points found but the quantizer is not fitted");
      if (Error e2 = CErr(sdb_index_set_codes(h_, qid.size(), qid.data(), qdata.data()), "could not load quantized points")) return e2;
    }
    // a point with codes does not load its raw vector (binary.go:283-290, product.go:357-365);
    // node 1 goes through sdb_index_set_start
    std::vector<uint8_t> has_q;
    for (uint64_t id : qid) {
      if (id >= has_q.size()) has_q.resize(id + 1, 0);
      has_q[id] = 1;
    }
    std::vector<uint64_t> vid2;
    std::vector<float> vdata2;
    for (size_t i = 0; i < vid.size(); ++i) {
      const uint64_t id = vid[i];
      if (id < has_q.size() && has_q[id]) continue;
      if (id == STARTID) {
        if (Error e2 = CErr(sdb_index_set_start(h_, &vdata[i * size_t(dim)]), "could not load start node")) return e2;
        continue;
      }
      vid2.push_back(id);
      vdata2.insert(vdata2.end(), vdata.begin() + i * size_t(dim), vdata.begin() + (i + 1) * size_t(dim));
    }
    if (!vid2.empty())
      if (Error e2 = CErr(sdb_index_set_vectors(h_, vid2.size(), vid2.data(), vdata2.data()), "could not load vectors")) return e2;
    for (uint64_t id : vid) SetAlive(id, true);
    for (uint64_t id : qid) SetAlive(id, true);
    // edges: first R of a list go to the adjacency row; the start node may own more (prune.go:137-151)
    const uint32_t R = uint32_t(params_.DegreeBound);
    std::vector<uint64_t> ids2, flat, overflow;
    std::vector<uint32_t> degs;
    for (size_t i = 0; i < eid.size(); ++i) {
      if (!Alive(eid[i])) continue;  // edges without a vector: cache.ErrNotFound on access in the reference
      const std::vector<uint64_t>& l = elists[i];
      size_t take = l.size();
      if (take > R) {
        if (eid[i] != STARTID) return Error("node " + std::to_string(eid[i]) + " has more edges than the degree bound");
        overflow.assign(l.begin() + R, l.end());
        take = R;
      }
      ids2.push_back(eid[i]);
      degs.push_back(uint32_t(take));
      flat.insert(flat.end(), l.begin(), l.begin() + take);
    }
    if (!ids2.empty())
      if (Error e2 = CErr(sdb_index_set_edges(h_, ids2.size(), ids2.data(), degs.data(), flat.data()), "could not load edges")) return e2;
    if (!overflow.empty())
      if (Error e2 = CErr(sdb_index_set_start_overflow(h_, overflow.size(), overflow.data()), "could not load start node edges")) return e2;
    // hydrated state is clean
    uint64_t n_dirty = 0;
    std::vector<uint64_t> scratch(sdb_index_max_node_id(h_) + 2);
    if (Error e2 = CErr(sdb_index_dirty_edges(h_, scratch.size(), scratch.data(), &n_dirty, 1), "could not reset dirty state")) return e2;
    const uint64_t dev_max = sdb_index_max_node_id(h_);
    if (dev_max > max_node_id_) max_node_id_ = dev_max;
    return Ok();
  }

  // setupStartNode (vamana.go:93-120)
  Error SetupStartNode() {
    if (Alive(STARTID)) return Ok();
    const uint32_t dim = params_.VectorSize;
    std::vector<float> v(dim);
    std::uniform_real_distribution<float> u(0.0f, 1.0f);
    float sum = 0.0f;
    for (uint32_t i = 0; i < dim; ++i) {
      v[i] = u(rng_) * 2 - 1;
      sum += v[i] * v[i];
    }
    const float norm = 1 / float(std::sqrt(double(sum)));
    for (uint32_t i = 0; i < dim; ++i) v[i] *= norm;
    if (Error e = CErr(sdb_index_set_start(h_, v.data()), "could not set start point")) return e;
    SetAlive(STARTID, true);
    dirty_vec_.push_back(STARTID);
    start_edges_dirty_ = true;  // nodeStore.Put(STARTID, ...) (vamana.go:118)
    if (max_node_id_ < STARTID) max_node_id_ = STARTID;
    return Ok();
  }

  // VectorStore.Flush for the three stores (plain.go:99-101, binary.go:236-244, product.go:307-320)
  Error FlushVectors() {
    const uint32_t dim = params_.VectorSize;
    std::vector<uint64_t> ids;
    if (all_vec_dirty_) {
      for (uint64_t id = 0; id < alive_.size(); ++id)
        if (alive_[id]) ids.push_back(id);
    } else {
      ids = dirty_vec_;
      std::sort(ids.begin(), ids.end());
      ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
      ids.erase(std::remove_if(ids.begin(), ids.end(), [&](uint64_t id) { return !Alive(id); }), ids.end());
    }
    for (uint64_t id : deleted_) {  // DeleteFrom (plain.go:141-146, binary.go:311-320, product.go:384-393)
      if (Alive(id)) continue;      // deleted and re-inserted later in the same session
      if (Error e = bucket_->Delete(conversion::NodeKey(id, 'v'))) return e;
      if (quant_kind_ != SDB_QUANT_NONE)
        if (Error e = bucket_->Delete(conversion::NodeKey(id, 'q'))) return e;
    }
    const size_t chunk = 65536;
    const bool write_codes = quant_kind_ != SDB_QUANT_NONE && quant_fitted_;
    // binary: codes replace the raw vector on disk (binary.go:298-309); product: both (product.go:373-382)
    const bool write_raw = !(quant_kind_ == SDB_QUANT_BINARY && quant_fitted_);
    const size_t cw = CodeWidth();
    std::vector<float> vbuf;
    std::vector<uint8_t> cbuf;
    for (size_t s = 0; s < ids.size(); s += chunk) {
      const size_t m = std::min(chunk, ids.size() - s);
      if (write_raw) {
        vbuf.resize(m * size_t(dim));
        if (Error e = CErr(sdb_index_get_vectors(h_, m, ids.data() + s, vbuf.data()), "could not read vectors")) return e;
        for (size_t i = 0; i < m; ++i)
          if (Error e = bucket_->Put(conversion::NodeKey(ids[s + i], 'v'), conversion::Float32ToBytes(&vbuf[i * size_t(dim)], dim)))
            return e.Wrap("could not write point vector");
      }
      if (write_codes) {
        cbuf.resize(m * cw);
        if (Error e = CErr(sdb_index_get_codes(h_, m, ids.data() + s, cbuf.data()), "could not read codes")) return e;
        for (size_t i = 0; i < m; ++i)
          if (Error e = bucket_->Put(conversion::NodeKey(ids[s + i], 'q'),
                                     std::string(reinterpret_cast<const char*>(&cbuf[i * cw]), cw)))
            return e.Wrap("could not write quantized point");
      }
    }
    if (quant_kind_ == SDB_QUANT_BINARY && quant_fitted_) {
      std::vector<float> thr(dim);
      if (Error e = CErr(sdb_index_get_bq_threshold(h_, thr.data()), "could not read binary quantizer threshold")) return e;
      if (Error e = bucket_->Put(binaryQuantizerThresholdKey, conversion::Float32ToBytes(thr))) return e;
    }
    if (quant_kind_ == SDB_QUANT_PRODUCT && quant_fitted_ && all_vec_dirty_) {
      std::vector<float> fc(size_t(pqM_) * pqK_ * (dim / pqM_)), cd(size_t(pqM_) * pqK_ * pqK_);
      if (Error e = CErr(sdb_index_get_pq(h_, fc.data(), cd.data()), "could not read product quantizer")) return e;
      if (Error e = bucket_->Put(productQuantizerCentroidDistsKey, conversion::Float32ToBytes(cd))) return e;
      if (Error e = bucket_->Put(productQuantizerFlatCentroidsKey, conversion::Float32ToBytes(fc))) return e;
    }
    dirty_vec_.clear();
    all_vec_dirty_ = false;
    return Ok();
  }

  // nodeStore.Flush (itemcache.go:236): rewrite dirty edge lists, drop deleted nodes
  Error FlushEdges() {
    const uint32_t R = uint32_t(params_.DegreeBound);
    for (uint64_t id : deleted_) {
      if (Alive(id)) continue;
      if (Error e = bucket_->Delete(conversion::NodeKey(id, 'e'))) return e.Wrap("could not delete vector");  // node.go:130-135
    }
    deleted_.clear();
    uint64_t n = 0;
    std::vector<uint64_t> ids(sdb_index_max_node_id(h_) + 2);
    if (Error e = CErr(sdb_index_dirty_edges(h_, ids.size(), ids.data(), &n, 1), "could not list dirty nodes")) return e;
    ids.resize(n);
    if (start_edges_dirty_ && std::find(ids.begin(), ids.end(), STARTID) == ids.end()) ids.insert(ids.begin(), STARTID);
    start_edges_dirty_ = false;
    ids.erase(std::remove_if(ids.begin(), ids.end(), [&](uint64_t id) { return !Alive(id); }), ids.end());
    const size_t chunk = 65536;
    std::vector<uint32_t> deg;
    std::vector<uint64_t> e;
    for (size_t s = 0; s < ids.size(); s += chunk) {
      const size_t m = std::min(chunk, ids.size() - s);
      deg.resize(m);
      e.resize(m * size_t(R));
      if (Error er = CErr(sdb_index_get_edges(h_, m, ids.data() + s, deg.data(), e.data()), "could not read edges")) return er;
      for (size_t i = 0; i < m; ++i) {
        std::vector<uint64_t> list(e.begin() + i * size_t(R), e.begin() + i * size_t(R) + deg[i]);
        if (ids[s + i] == STARTID) {
          uint64_t no = 0;
          sdb_index_get_start_overflow(h_, 0, nullptr, &no);
          if (no) {
            std::vector<uint64_t> extra(no);
            if (Error er = CErr(sdb_index_get_start_overflow(h_, no, extra.data(), &no), "could not read start node edges")) return er;
            list.insert(list.end(), extra.begin(), extra.end());
          }
        }
        if (Error er = bucket_->Put(conversion::NodeKey(ids[s + i], 'e'), conversion::EdgeListToBytes(list)))
          return er.Wrap("could not write edges");  // node.go:122-128
      }
    }
    return Ok();
  }

  std::string name_;
  models::IndexVectorVamanaParameters params_;
  diskstore::Bucket* bucket_ = nullptr;
  sdb_index* h_ = nullptr;
  std::mt19937_64 rng_;
  std::mutex write_mu_;
  uint64_t max_node_id_ = 0;
  int quant_kind_ = SDB_QUANT_NONE;
  bool quant_fitted_ = false;
  uint32_t pqM_ = 0, pqK_ = 0;
  std::vector<uint8_t> alive_;
  std::vector<uint64_t> dirty_vec_, deleted_;
  bool all_vec_dirty_ = false;
  bool start_edges_dirty_ = false;
};

}  // namespace vamana
}  // namespace semadb
