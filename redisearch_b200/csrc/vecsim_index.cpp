// Host logic of the B200 FLAT index.  See vecsim_index.h for the reference files mirrored.
#include "vecsim_index.h"
#include "host_numeric.h"
#include "topk_common.cuh"
#include "coarse_tc.h"
#include "micro_batcher.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <limits>
#include <thread>

namespace rsb200 {

Globals &globals() {
    static Globals g;
    return g;
}

#define CU_OK(expr)                                                                                 \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            fprintf(stderr, "[vecsim_b200] CUDA error %s at %s:%d: %s\n", cudaGetErrorName(_e), __FILE__, __LINE__,  \
                    cudaGetErrorString(_e));                                                        \
            return false;                                                                           \
        }                                                                                           \
    } while (0)

// ------------------------------------------------------------------------------------------------
// QueryCtx
// ------------------------------------------------------------------------------------------------
QueryCtx::~QueryCtx() {
    if (stream) cudaStreamSynchronize(stream);
    cudaFree(d_query);
    cudaFreeHost(h_query);
    cudaFree(d_cand);
    cudaFree(d_out);
    cudaFreeHost(h_out);
    cudaFree(d_scores);
    cudaFree(d_count);
    cudaFreeHost(h_count);
    cudaFreeHost(h_abort);
    cudaFree(d_ids);
    cudaFreeHost(h_ids);
    cudaFree(d_dist);
    cudaFreeHost(h_dist);
    if (ev_start) cudaEventDestroy(ev_start);
    if (ev_stop) cudaEventDestroy(ev_stop);
    if (stream) cudaStreamDestroy(stream);
}
bool QueryCtx::init() {
    CU_OK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CU_OK(cudaEventCreate(&ev_start));
    CU_OK(cudaEventCreate(&ev_stop));
    CU_OK(cudaMalloc(&d_count, 16));
    CU_OK(cudaMallocHost(&h_count, 16));
    CU_OK(cudaHostAlloc(&h_abort, 64, cudaHostAllocMapped));
    *h_abort = 0;
    void *dp = nullptr;
    CU_OK(cudaHostGetDevicePointer(&dp, h_abort, 0));
    d_abort = static_cast<const uint32_t *>(dp);
    return true;
}
bool QueryCtx::need_query(size_t bytes) {
    if (bytes <= query_cap) return true;
    cudaStreamSynchronize(stream);
    cudaFree(d_query);
    cudaFreeHost(h_query);
    d_query = nullptr;
    h_query = nullptr;
    query_cap = 0;
    const size_t cap = std::max<size_t>(bytes, 64 * 1024);
    CU_OK(cudaMalloc(&d_query, cap));
    CU_OK(cudaMallocHost(&h_query, cap));
    query_cap = cap;
    return true;
}
bool QueryCtx::need_cand(size_t elems) {
    if (elems <= cand_cap) return true;
    cudaStreamSynchronize(stream);
    cudaFree(d_cand);
    d_cand = nullptr;
    cand_cap = 0;
    const size_t cap = std::max<size_t>(elems, 64 * 1024);
    CU_OK(cudaMalloc(&d_cand, cap * sizeof(uint64_t)));
    cand_cap = cap;
    return true;
}
bool QueryCtx::need_out(size_t elems) {
    if (elems <= out_cap) return true;
    cudaStreamSynchronize(stream);
    cudaFree(d_out);
    cudaFreeHost(h_out);
    d_out = nullptr;
    h_out = nullptr;
    out_cap = 0;
    const size_t cap = std::max<size_t>(elems, 4096);
    CU_OK(cudaMalloc(&d_out, cap * sizeof(uint64_t)));
    CU_OK(cudaMallocHost(&h_out, cap * sizeof(uint64_t)));
    out_cap = cap;
    return true;
}
bool QueryCtx::need_scores(size_t n) {
    if (n <= scores_cap) return true;
    cudaStreamSynchronize(stream);
    cudaFree(d_scores);
    d_scores = nullptr;
    scores_cap = 0;
    const size_t cap = n + n / 8 + 1024;
    CU_OK(cudaMalloc(&d_scores, cap * sizeof(float)));
    scores_cap = cap;
    return true;
}
bool QueryCtx::need_ids(size_t n) {
    if (n <= ids_cap) return true;
    cudaStreamSynchronize(stream);
    cudaFree(d_ids);
    cudaFreeHost(h_ids);
    cudaFree(d_dist);
    cudaFreeHost(h_dist);
    d_ids = h_ids = nullptr;
    d_dist = h_dist = nullptr;
    ids_cap = 0;
    const size_t cap = std::max<size_t>(n, 1024);
    CU_OK(cudaMalloc(&d_ids, cap * 4));
    CU_OK(cudaMallocHost(&h_ids, cap * 4));
    CU_OK(cudaMalloc(&d_dist, cap * 4));
    CU_OK(cudaMallocHost(&h_dist, cap * 4));
    ids_cap = cap;
    return true;
}

// ------------------------------------------------------------------------------------------------
// construction
// ------------------------------------------------------------------------------------------------
static size_t elem_size(VecSimType t) {
    switch (t) {
    case VecSimType_FLOAT32: return 4;
    case VecSimType_FLOAT16:
    case VecSimType_BFLOAT16: return 2;
    case VecSimType_INT8:
    case VecSimType_UINT8: return 1;
    default: return 0;
    }
}

void FlatIndex::log(const char *level, const char *fmt, ...) const {
    logCallbackFunction cb = globals().log_cb.load();
    if (!cb) return;
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    cb(log_ctx_, level, buf);
}

FlatIndex *FlatIndex::create(const BFParams &p, void *log_ctx) {
    const size_t es = elem_size(p.type);
    if (es == 0 || p.dim == 0) return nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        logCallbackFunction cb = globals().log_cb.load();
        const char *msg = "vecsim_b200: no CUDA device available; this library has no CPU fallback";
        if (cb)
            cb(log_ctx, "warning", msg);
        else
            fprintf(stderr, "%s\n", msg);
        cudaGetLastError();
        return nullptr;
    }
    std::unique_ptr<FlatIndex> ix(new FlatIndex());
    ix->type_ = p.type;
    ix->metric_ = p.metric;
    ix->dim_ = p.dim;
    ix->multi_ = p.multi;
    ix->block_size_ = p.blockSize ? p.blockSize : DEFAULT_BLOCK_SIZE;
    ix->log_ctx_ = log_ctx;
    ix->elem_bytes_ = es;
    switch (p.type) {
    case VecSimType_FLOAT32: ix->dtype_ = DT_F32; break;
    case VecSimType_FLOAT16: ix->dtype_ = DT_F16; break;
    case VecSimType_BFLOAT16: ix->dtype_ = DT_BF16; break;
    case VecSimType_INT8: ix->dtype_ = DT_I8; break;
    default: ix->dtype_ = DT_U8; break;
    }
    const bool is_int = (ix->dtype_ == DT_I8 || ix->dtype_ == DT_U8);
    ix->mkind_ = (p.metric == VecSimMetric_L2) ? MT_L2 : (p.metric == VecSimMetric_IP || !is_int) ? MT_IP : MT_COS;
    ix->stored_bytes_ = p.dim * es + ((is_int && p.metric == VecSimMetric_Cosine) ? sizeof(float) : 0);
    // fp32 rows are read with 4-byte lane loads (any dim); the narrower types with 16-byte vectors.
    ix->pitch_ = (ix->dtype_ == DT_F32) ? ix->stored_bytes_ : ((ix->stored_bytes_ + 15) & ~(size_t)15);
    if (cudaStreamCreateWithFlags(&ix->copy_stream_, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    // pinned staging: up to 32 MiB of appended rows between flushes
    ix->stage_cap_rows_ = std::max<size_t>(1, std::min<size_t>((32u << 20) / ix->pitch_, 1u << 20));
    if (cudaMallocHost(&ix->h_stage_, ix->stage_cap_rows_ * ix->pitch_) != cudaSuccess) return nullptr;
    memset(ix->h_stage_, 0, ix->stage_cap_rows_ * ix->pitch_);
    if (p.initialCapacity && !ix->reserve(p.initialCapacity)) return nullptr;
    return ix.release();
}

FlatIndex::~FlatIndex() {
    {
        std::lock_guard<std::mutex> g(pool_mu_);
        pool_.clear();
    }
    if (copy_stream_) {
        cudaStreamSynchronize(copy_stream_);
        cudaStreamDestroy(copy_stream_);
    }
    cudaFree(d_rows_);
    cudaFree(d_shadow_);
    cudaFree(d_norm2_);
    cudaFree(d_stats_);
    cudaFree(d_label_to_id_);
    cudaFree(d_id_to_label_);
    cudaFreeHost(h_stage_);
}

CorpusView FlatIndex::view() const {
    CorpusView v;
    v.rows = d_rows_;
    v.pitch = pitch_;
    v.n_rows = (uint32_t)count_;
    v.dim = (uint32_t)dim_;
    v.dtype = dtype_;
    v.metric = mkind_;
    return v;
}

std::unique_ptr<QueryCtx> FlatIndex::checkout() {
    {
        std::unique_lock<std::mutex> g(pool_mu_);
        if (!pool_.empty()) {
            auto c = std::move(pool_.back());
            pool_.pop_back();
            g.unlock();
            if (c->abandoned) { // its last user timed out and left: let that work drain before the buffers are reused
                cudaStreamSynchronize(c->stream);
                c->abandoned = false;
                *c->h_abort = 0;
            }
            return c;
        }
    }
    std::unique_ptr<QueryCtx> c(new QueryCtx());
    if (!c->init()) return nullptr;
    return c;
}
void FlatIndex::checkin(std::unique_ptr<QueryCtx> c) {
    if (!c) return;
    std::lock_guard<std::mutex> g(pool_mu_);
    if (pool_.size() < 64) pool_.push_back(std::move(c));
}

bool FlatIndex::timed_out(void *ctx) const {
    timeoutCallbackFunction cb = globals().timeout_cb.load();
    return cb && cb(ctx) != 0;
}

int FlatIndex::wait_polling(cudaStream_t s, void *timeout_ctx) const {
    timeoutCallbackFunction cb = globals().timeout_cb.load();
    if (!cb) return cudaStreamSynchronize(s) == cudaSuccess ? 0 : -1;
    for (;;) {
        const cudaError_t e = cudaStreamQuery(s);
        if (e == cudaSuccess) return 0;
        if (e != cudaErrorNotReady) return -1;
        if (cb(timeout_ctx) != 0) return 1;
        std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
}

// ------------------------------------------------------------------------------------------------
// preprocessing (VS/spaces/computer/preprocessors.h:49-146)
// ------------------------------------------------------------------------------------------------
void FlatIndex::preprocess_storage(const void *blob, uint8_t *dst) const {
    memcpy(dst, blob, dim_ * elem_bytes_);
    if (metric_ != VecSimMetric_Cosine) return;
    switch (dtype_) {
    case DT_F32: normalize_f32(reinterpret_cast<float *>(dst), dim_); break;
    case DT_F16: normalize_f16(reinterpret_cast<uint16_t *>(dst), dim_); break;
    case DT_BF16: normalize_bf16(reinterpret_cast<uint16_t *>(dst), dim_); break;
    case DT_I8: append_int_norm(reinterpret_cast<int8_t *>(dst), dim_); break;
    case DT_U8: append_int_norm(reinterpret_cast<uint8_t *>(dst), dim_); break;
    }
}
void FlatIndex::preprocess_query(const void *blob, uint8_t *dst) const { preprocess_storage(blob, dst); }

// ------------------------------------------------------------------------------------------------
// storage
// ------------------------------------------------------------------------------------------------
bool FlatIndex::grow_to(size_t rows) {
    if (rows <= capacity_) return true;
    size_t cap = std::max(rows, capacity_ + capacity_ / 2);
    cap = ((cap + block_size_ - 1) / block_size_) * block_size_;
    uint8_t *nu = nullptr;
    cudaError_t e = cudaMalloc(&nu, cap * pitch_);
    if (e != cudaSuccess && cap > rows) { // retry with the exact size
        cudaGetLastError();
        cap = ((rows + block_size_ - 1) / block_size_) * block_size_;
        e = cudaMalloc(&nu, cap * pitch_);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        log("warning", "vecsim_b200: cannot allocate %zu bytes of HBM", cap * pitch_);
        return false;
    }
    if (resident_) {
        CU_OK(cudaMemcpyAsync(nu, d_rows_, resident_ * pitch_, cudaMemcpyDeviceToDevice, copy_stream_));
        CU_OK(cudaStreamSynchronize(copy_stream_));
    }
    cudaFree(d_rows_);
    d_rows_ = nu;
    capacity_ = cap;
    return true;
}

bool FlatIndex::reserve(size_t rows) {
    std::lock_guard<std::mutex> g(mu_);
    if (id_to_label_.capacity() < rows) id_to_label_.reserve(rows);
    return grow_to(rows);
}

// caller holds mu_
static bool flush_locked(uint8_t *d_rows, size_t pitch, uint8_t *h_stage, size_t &resident, size_t count,
                         cudaStream_t s) {
    if (resident == count) return true;
    const size_t n = count - resident;
    CU_OK(cudaMemcpyAsync(d_rows + resident * pitch, h_stage, n * pitch, cudaMemcpyHostToDevice, s));
    CU_OK(cudaStreamSynchronize(s));
    resident = count;
    return true;
}

bool FlatIndex::flush() {
    std::lock_guard<std::mutex> g(mu_);
    return flush_locked(d_rows_, pitch_, h_stage_, resident_, count_, copy_stream_);
}

int FlatIndex::add(const void *blob, size_t label) {
    std::lock_guard<std::mutex> g(mu_);
    if (!multi_) {
        auto it = label_to_id_.find(label);
        if (it != label_to_id_.end()) {
            // brute_force_single.h:139-144: overwrite in place with the RAW blob (the reference does
            // not re-run the storage preprocessor here).  For int8/uint8 cosine the reference reads
            // 4 bytes past the caller's blob; we recompute the norm instead of reading out of bounds.
            const idType id = it->second;
            std::vector<uint8_t> tmp(pitch_, 0);
            memcpy(tmp.data(), blob, dim_ * elem_bytes_);
            if (mkind_ == MT_COS) {
                if (dtype_ == DT_I8)
                    append_int_norm(reinterpret_cast<int8_t *>(tmp.data()), dim_);
                else
                    append_int_norm(tmp.data(), dim_);
            }
            if (id >= resident_) {
                memcpy(h_stage_ + (id - resident_) * pitch_, tmp.data(), pitch_);
            } else {
                if (cudaMemcpy(d_rows_ + (size_t)id * pitch_, tmp.data(), pitch_, cudaMemcpyHostToDevice) != cudaSuccess)
                    return 0;
                if (d_shadow_) shadow_dirty_.push_back(id);
            }
            // the overwritten row is the caller's RAW blob: a cosine index may now hold a non-unit row, so the coarse
            // proof must stop assuming unit vectors (it switches to the norm-scaled bound of the inner-product route)
            if (metric_ == VecSimMetric_Cosine && dtype_ == DT_F32 && !raw_rows_) {
                raw_rows_ = true;
                shadow_rows_ = 0; // |row|^2 and the running maxima have to be built for every row
                shadow_dirty_.clear();
            }
            return 0;
        }
    }
    if (count_ >= (size_t)std::numeric_limits<uint32_t>::max() - 1) return 0;
    if (count_ - resident_ >= stage_cap_rows_) {
        if (!grow_to(count_ + 1)) return 0;
        if (!flush_locked(d_rows_, pitch_, h_stage_, resident_, count_, copy_stream_)) return 0;
    }
    if (!grow_to(count_ + 1)) return 0;
    uint8_t *slot = h_stage_ + (count_ - resident_) * pitch_;
    preprocess_storage(blob, slot);
    const idType id = (idType)count_++;
    id_to_label_.push_back(label);
    if (multi_)
        label_to_ids_[label].push_back(id);
    else
        label_to_id_[label] = id;
    labels_dirty_ = true;
    l2i_dirty_ = true;
    return 1;
}

int FlatIndex::add_bulk(const void *blobs, size_t stride, size_t n, const size_t *labels, size_t label0) {
    int added = 0;
    for (size_t i = 0; i < n; i++)
        added += add(static_cast<const uint8_t *>(blobs) + i * stride, labels ? labels[i] : label0 + i);
    return added;
}

int FlatIndex::add_bulk_device(const void *d_src, size_t n, size_t label0) {
    std::lock_guard<std::mutex> g(mu_);
    if (n == 0) return 0;
    if (!flush_locked(d_rows_, pitch_, h_stage_, resident_, count_, copy_stream_)) return -1;
    if (!grow_to(count_ + n)) return -1;
    if (cudaMemcpyAsync(d_rows_ + count_ * pitch_, d_src, n * pitch_, cudaMemcpyDeviceToDevice, copy_stream_) !=
            cudaSuccess ||
        cudaStreamSynchronize(copy_stream_) != cudaSuccess)
        return -1;
    id_to_label_.reserve(count_ + n);
    for (size_t i = 0; i < n; i++) {
        const idType id = (idType)(count_ + i);
        id_to_label_.push_back(label0 + i);
        if (multi_)
            label_to_ids_[label0 + i].push_back(id);
        else
            label_to_id_[label0 + i] = id;
    }
    count_ += n;
    resident_ = count_;
    labels_dirty_ = true;
    l2i_dirty_ = true;
    return (int)n;
}

int FlatIndex::remove(size_t label) {
    std::lock_guard<std::mutex> g(mu_);
    std::vector<idType> victims;
    if (multi_) {
        auto it = label_to_ids_.find(label);
        if (it == label_to_ids_.end()) return 0;
        victims = it->second;
        label_to_ids_.erase(it);
    } else {
        auto it = label_to_id_.find(label);
        if (it == label_to_id_.end()) return 0;
        victims.push_back(it->second);
        label_to_id_.erase(it);
    }
    if (!flush_locked(d_rows_, pitch_, h_stage_, resident_, count_, copy_stream_)) return 0;
    // brute_force.h:196-224 — move the last row into the hole; with several victims process them
    // one by one (brute_force_multi.h:143-165), re-reading ids that a previous swap relocated.
    int removed = 0;
    std::sort(victims.begin(), victims.end(), std::greater<idType>());
    for (idType id : victims) {
        const idType last = (idType)(count_ - 1);
        if (id != last) {
            const size_t last_label = id_to_label_[last];
            cudaMemcpyAsync(d_rows_ + (size_t)id * pitch_, d_rows_ + (size_t)last * pitch_, pitch_,
                            cudaMemcpyDeviceToDevice, copy_stream_);
            if (d_shadow_) shadow_dirty_.push_back(id);
            id_to_label_[id] = last_label;
            if (multi_) {
                auto &v = label_to_ids_[last_label];
                for (auto &x : v)
                    if (x == last) x = id;
            } else {
                label_to_id_[last_label] = id;
            }
        }
        id_to_label_.pop_back();
        count_--;
        removed++;
    }
    // row ids >= count_ will be re-used by later appends: the shadow copy (and |row|^2) of those ids is stale
    shadow_rows_ = std::min(shadow_rows_, count_);
    cudaStreamSynchronize(copy_stream_);
    resident_ = count_;
    labels_dirty_ = true;
    l2i_dirty_ = true;
    return removed;
}

bool FlatIndex::read_rows(size_t first, size_t n, void *host_dst) {
    if (!flush()) return false;
    if (first + n > count_ || !host_dst) return false;
    if (n == 0) return true;
    return cudaMemcpy2D(host_dst, stored_bytes_, d_rows_ + first * pitch_, pitch_, stored_bytes_, n, cudaMemcpyDeviceToHost) == cudaSuccess;
}

bool FlatIndex::sync_labels_to_device() {
    std::lock_guard<std::mutex> g(mu_);
    if (!labels_dirty_ && d_id_to_label_) return true;
    if (count_ > d_labels_cap_) {
        cudaFree(d_id_to_label_);
        d_id_to_label_ = nullptr;
        const size_t cap = std::max(capacity_, count_);
        CU_OK(cudaMalloc(&d_id_to_label_, cap * sizeof(uint64_t)));
        d_labels_cap_ = cap;
    }
    static_assert(sizeof(size_t) == sizeof(uint64_t), "labels are 64-bit");
    if (count_)
        CU_OK(cudaMemcpy(d_id_to_label_, id_to_label_.data(), count_ * sizeof(uint64_t), cudaMemcpyHostToDevice));
    labels_dirty_ = false;
    return true;
}

// ------------------------------------------------------------------------------------------------
// queries
// ------------------------------------------------------------------------------------------------
bool FlatIndex::upload_query(QueryCtx &c, const uint8_t *stored_q, size_t nq) {
    const size_t qp = (stored_bytes_ + 15) & ~(size_t)15;
    if (!c.need_query(qp * nq)) return false;
    if (stored_q != c.h_query) {
        for (size_t i = 0; i < nq; i++) {
            memcpy(c.h_query + i * qp, stored_q + i * stored_bytes_, stored_bytes_);
            memset(c.h_query + i * qp + stored_bytes_, 0, qp - stored_bytes_);
        }
    }
    CU_OK(cudaMemcpyAsync(c.d_query, c.h_query, qp * nq, cudaMemcpyHostToDevice, c.stream));
    return true;
}

namespace {
struct KeyedResult {
    uint32_t key;
    size_t label;
};
} // namespace

// reply ordering: (score asc, label asc) — the order the reference's heap drains in
// (vecsim_stl.h:64-84) — or by label (vec_utils.cpp:100-103).
void FlatIndex::finish_reply(VecSimQueryReply *rep, VecSimQueryReply_Order order) const {
    auto &r = rep->results;
    if (order == BY_ID) {
        std::sort(r.begin(), r.end(), [](const VecSimQueryResult &a, const VecSimQueryResult &b) { return a.id < b.id; });
    } else {
        std::sort(r.begin(), r.end(), [](const VecSimQueryResult &a, const VecSimQueryResult &b) {
            const bool an = std::isnan(a.score), bn = std::isnan(b.score);
            if (an != bn) return bn; // NaN last
            if (!an && a.score != b.score) return a.score < b.score;
            return a.id < b.id;
        });
    }
}

long FlatIndex::select_from_scores(QueryCtx &c, uint32_t n, bool has_cursor, uint64_t cursor, size_t want) {
    if (want == 0 || n == 0) return 0;
    if (!c.need_out(want + 1)) return -1;
    LaunchCounters lc;
    const uint64_t *cur_ptr = nullptr;
    if (has_cursor) {
        *reinterpret_cast<uint64_t *>(c.h_count) = cursor;
        if (cudaMemcpyAsync(c.d_out + want, c.h_count, 8, cudaMemcpyHostToDevice, c.stream) != cudaSuccess) return -1;
        cur_ptr = c.d_out + want;
    }
    const uint32_t lists = plan_select_scores_lists(n);
    size_t found = 0;
    while (found < want) {
        const uint32_t chunk = (uint32_t)std::min<size_t>(kMaxFusedK, want - found);
        if (!c.need_cand((size_t)lists * chunk)) return -1;
        if (launch_select_scores(c.d_scores, n, cur_ptr, chunk, c.d_cand, c.stream, &lc) != cudaSuccess) return -1;
        if (launch_final_select(c.d_cand, 1, lists * chunk, chunk, c.d_out + found, c.stream, &lc) != cudaSuccess)
            return -1;
        found += chunk;
        cur_ptr = c.d_out + found - 1;
    }
    if (cudaMemcpyAsync(c.h_out, c.d_out, want * 8, cudaMemcpyDeviceToHost, c.stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(c.stream) != cudaSuccess) return -1;
    launches_total_ += lc.launches;
    size_t real = 0;
    while (real < want && c.h_out[real] != kEmptySlot) real++;
    return (long)real;
}

VecSimQueryReply *FlatIndex::topk(const void *q, size_t k, VecSimQueryParams *qp, VecSimQueryReply_Order order) {
    auto *rep = new VecSimQueryReply();
    last_mode_ = STANDARD_KNN;
    void *tctx = qp ? qp->timeoutCtx : nullptr;
    if (k == 0) return rep; // brute_force.h:251-253
    if (!flush()) return rep;
    const size_t n = count_;
    if (n == 0) return rep;
    if (timed_out(tctx)) {
        rep->code = VecSim_QueryReply_TimedOut;
        return rep;
    }
    auto c = checkout();
    if (!c) return rep;
    const size_t qpitch = (stored_bytes_ + 15) & ~(size_t)15;
    bool ok = c->need_query(qpitch);
    if (ok) {
        memset(c->h_query, 0, qpitch);
        preprocess_query(q, c->h_query);
        ok = upload_query(*c, c->h_query, 1);
    }
    const CorpusView v = view();
    LaunchCounters lc;
    if (ok && !multi_ && std::min(k, n) <= (size_t)kMaxFusedK) {
        const uint32_t ke = (uint32_t)std::min(k, n);
        const uint64_t *d_res = nullptr;
        if (single_query_takes_coarse(ke)) {
            // an up-to-date fp16 shadow exists (a batch built it): one pass over 15 GB of it + exact rescoring + proof
            // beats the 31 GB exact scan; same answer (DESIGN.md §4)
            uint64_t *r = nullptr;
            ok = batch_scan(*c, c->d_query, qpitch, 1, ke, c->stream, lc, &r);
            d_res = r;
        } else {
            last_batch_path_ = 0;
            const ScanPlan plan = plan_scan_topk(v, 1, ke);
            ok = c->need_cand(plan.cand_elems) && c->need_out(ke);
            if (ok) {
                cudaEventRecord(c->ev_start, c->stream);
                ok = launch_scan_topk(v, c->d_query, qpitch, 1, ke, plan, c->d_cand, c->stream, &lc, nullptr, c->d_abort) == cudaSuccess;
                cudaEventRecord(c->ev_stop, c->stream);
            }
            ok = ok && launch_final_select(c->d_cand, 1, plan.lists_per_query * ke, ke, c->d_out, c->stream, &lc) == cudaSuccess;
            d_res = c->d_out;
        }
        ok = ok && cudaMemcpyAsync(c->h_out, d_res, ke * 8, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess;
        if (ok) {
            const int w = wait_polling(c->stream, tctx);
            if (w == 1) { // deadline passed while the scan was running
                c->abandoned = true;
                *c->h_abort = 1; // the kernels still running on its stream wind down
                launches_total_ += lc.launches;
                checkin(std::move(c));
                rep->code = VecSim_QueryReply_TimedOut;
                return rep;
            }
            ok = w == 0;
        }
        if (ok) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, c->ev_start, c->ev_stop) == cudaSuccess) {
                std::lock_guard<std::mutex> g(stats_mu_);
                scan_us_ += ms * 1000.0;
                scan_launches_++;
                scan_bytes_ += (uint64_t)n * stored_bytes_;
            }
            for (uint32_t i = 0; i < ke; i++) {
                const uint64_t comp = c->h_out[i];
                if (comp == kEmptySlot) break;
                rep->results.push_back({id_to_label_[(uint32_t)comp], (double)key_to_float((uint32_t)(comp >> 32))});
            }
        }
    } else if (ok) {
        // k > kMaxFusedK or multi-value: materialise all scores, then cursor-select in chunks.
        ok = c->need_scores(n);
        if (ok) {
            cudaEventRecord(c->ev_start, c->stream);
            ok = launch_scan_scores(v, c->d_query, c->d_scores, c->stream, &lc) == cudaSuccess;
            cudaEventRecord(c->ev_stop, c->stream);
        }
        if (ok) {
            const size_t want_labels = std::min(k, label_count());
            bool has_cursor = false;
            uint64_t cursor = 0;
            std::unordered_set<size_t> seen;
            size_t scanned = 0;
            while (ok && rep->results.size() < want_labels && scanned < n) {
                const size_t want = multi_ ? std::min<size_t>(std::max<size_t>(2 * (want_labels - rep->results.size()), 64), n - scanned)
                                           : std::min(want_labels - rep->results.size(), n - scanned);
                const long got = select_from_scores(*c, (uint32_t)n, has_cursor, cursor, want);
                if (got < 0) {
                    ok = false;
                    break;
                }
                for (long i = 0; i < got && rep->results.size() < want_labels; i++) {
                    const uint64_t comp = c->h_out[i];
                    const size_t label = id_to_label_[(uint32_t)comp];
                    if (multi_ && !seen.insert(label).second) continue; // best score per label comes first
                    rep->results.push_back({label, (double)key_to_float((uint32_t)(comp >> 32))});
                }
                scanned += (size_t)got;
                if ((size_t)got < want) break;
                has_cursor = true;
                cursor = c->h_out[got - 1];
            }
            float ms = 0;
            if (ok && cudaEventElapsedTime(&ms, c->ev_start, c->ev_stop) == cudaSuccess) {
                std::lock_guard<std::mutex> g(stats_mu_);
                scan_us_ += ms * 1000.0;
                scan_launches_++;
                scan_bytes_ += (uint64_t)n * stored_bytes_;
            }
        }
    }
    launches_total_ += lc.launches;
    if (!ok) {
        log("warning", "vecsim_b200: top-k query failed on device");
        rep->results.clear();
    }
    checkin(std::move(c));
    if (timed_out(tctx)) {
        rep->results.clear();
        rep->code = VecSim_QueryReply_TimedOut;
        return rep;
    }
    finish_reply(rep, order);
    return rep;
}

// -1 = from env VECSIM_B200_COARSE (default 1), 0 = exact scans only, 1 = fp16 shadow rows, 2 = TF32 on the fp32 rows
std::atomic<int> g_coarse_mode{-1};

// second tier of the coarse route (lists of 128 for the queries the first proof left open); VECSIM_B200_TIER2=0 turns it off
static bool coarse_tier2_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("VECSIM_B200_TIER2");
        v = (e && atoi(e) == 0) ? 0 : 1;
    }
    return v != 0;
}

// two-pass first tier of the fp16 route (sample pass -> fixed admission bound -> main pass); VECSIM_B200_FIXED=0 falls back
// to the single pass with adaptive lists
static bool coarse_fixed_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("VECSIM_B200_FIXED");
        v = (e && atoi(e) == 0) ? 0 : 1;
    }
    return v != 0;
}

static int coarse_mode() {
    int m = g_coarse_mode.load();
    if (m < 0) {
        const char *e = getenv("VECSIM_B200_COARSE");
        m = e ? atoi(e) : 1;
        if (m < 0 || m > 2) m = 1;
        g_coarse_mode.store(m);
    }
    return m;
}

// Single queries (and batches below 16) take the tensor-core route only if that costs nothing extra: mode 1, an fp16
// shadow that is already complete, fp32 cosine, k within the coarse lists.
bool FlatIndex::single_query_takes_coarse(uint32_t ke) {
    if (coarse_mode() != 1 || multi_ || coarse_disabled_ || dtype_ != DT_F32) return false;
    if (!unit_rows() && !(shadow_max_abs_ <= 60000.0f)) return false; // fp16 range (also false before the first build)
    {
        std::lock_guard<std::mutex> g(mu_);
        if (!d_shadow_ || shadow_rows_ != count_ || !shadow_dirty_.empty() || shadow_cap_ < count_) return false;
    }
    return coarse_supported(view(), 1, ke, CoarseF16);
}

// Bring the fp16 shadow copy of the rows up to date on `st` (rows appended, overwritten or moved by a
// swap-delete since the last coarse batch).  Returns false if HBM for the shadow cannot be had; the
// caller then runs the TF32 variant on the fp32 rows.
bool FlatIndex::ensure_shadow(cudaStream_t st) {
    std::lock_guard<std::mutex> g(mu_);
    if (shadow_cap_ < count_ || !d_shadow_) {
        const size_t cap = std::max(capacity_, count_);
        uint8_t *nu = nullptr;
        if (cudaMalloc(&nu, coarse_shadow_bytes((uint32_t)cap, (uint32_t)dim_)) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        cudaFree(d_shadow_); // rows are re-converted below; converting 10M x 768 takes ~7 ms
        d_shadow_ = nu;
        cudaFree(d_norm2_);
        d_norm2_ = nullptr;
        shadow_cap_ = cap;
        shadow_rows_ = 0;
        shadow_dirty_.clear();
    }
    if (!unit_rows() && !d_norm2_) { // L2 / raw inner product / cosine after a raw overwrite: the error bound (and the L2
                                     // epilogue) need |row|^2 of every row
        if (!d_stats_ && (cudaMalloc(&d_stats_, 8) != cudaSuccess || cudaMemset(d_stats_, 0, 8) != cudaSuccess)) {
            cudaGetLastError();
            return false;
        }
        if (cudaMalloc(&d_norm2_, shadow_cap_ * sizeof(float)) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        shadow_rows_ = 0;
        shadow_dirty_.clear();
    }
    if (shadow_rows_ > count_) shadow_rows_ = count_;
    bool launched = false;
    if (shadow_dirty_.size() > 256) {
        shadow_rows_ = 0;
        shadow_dirty_.clear();
    }
    for (idType id : shadow_dirty_)
        if (id < shadow_rows_) {
            if (launch_to_f16_tiled(d_rows_, pitch_, (uint32_t)dim_, id, 1, d_shadow_, st) != cudaSuccess) return false;
            if (d_norm2_ && launch_row_stats(d_rows_, pitch_, (uint32_t)dim_, id, 1, d_norm2_, d_stats_, st) != cudaSuccess) return false;
            launched = true;
        }
    shadow_dirty_.clear();
    if (shadow_rows_ < count_) {
        if (launch_to_f16_tiled(d_rows_, pitch_, (uint32_t)dim_, (uint32_t)shadow_rows_, (uint32_t)(count_ - shadow_rows_), d_shadow_,
                                st) != cudaSuccess)
            return false;
        if (d_norm2_ && launch_row_stats(d_rows_, pitch_, (uint32_t)dim_, (uint32_t)shadow_rows_, (uint32_t)(count_ - shadow_rows_), d_norm2_,
                                         d_stats_, st) != cudaSuccess)
            return false;
        shadow_rows_ = count_;
        launched = true;
    }
    // other query streams may read the shadow as soon as the lock is released
    if (launched) {
        uint32_t h[2] = {0, 0};
        if (d_norm2_ && cudaMemcpyAsync(h, d_stats_, 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) return false;
        if (cudaStreamSynchronize(st) != cudaSuccess) return false;
        if (d_norm2_) { // running maxima over every row ever converted (deletes do not lower them: conservative)
            float n2, ma;
            memcpy(&n2, &h[0], 4);
            memcpy(&ma, &h[1], 4);
            shadow_max_norm_ = std::sqrt(n2);
            shadow_max_abs_ = ma;
        }
    }
    return true;
}

// Enqueue on `st`: the `ke` best composites of each of `nq` device-resident stored-form queries into
// d_out [nq][ke].  Cosine fp32 batches take the tensor-core coarse pass + exact rescoring + proof, with
// the exact scan as an on-device fallback for unverified queries; everything else takes the exact
// fused scan.  ev_start/ev_stop of `c` bracket the dominant scan kernel.
bool FlatIndex::batch_scan(QueryCtx &c, const void *d_q, size_t qpitch, uint32_t nq, uint32_t ke, cudaStream_t st,
                           LaunchCounters &lc, uint64_t **d_result) {
    const CorpusView v = view();
    const ScanPlan sp = plan_scan_topk(v, nq, ke);
    const int cmode = coarse_mode();
    // fp16 / bf16 corpora: the tensor-core GEMM with fp32 accumulation IS the distance (within the 1e-2 bar by four
    // orders of magnitude), so the batch is one kernel + the usual final selection — no shadow, no rescoring
    const bool is16 = dtype_ == DT_F16 || dtype_ == DT_BF16, is8 = dtype_ == DT_I8 || dtype_ == DT_U8;
    const CoarseKind dkind = is16 ? CoarseDirect16 : CoarseDirect8;
    if (cmode != 0 && !multi_ && nq >= 16 && (is16 || is8) && coarse_supported(v, nq, ke, dkind)) {
        // int8 / uint8: kind::i8 dot products are exact integers and the epilogue applies the reference's own
        // float expression, so that route is bit-exact
        const CoarseOperands ops{v.rows, v.pitch, d_q, qpitch, (dtype_ == DT_BF16 || dtype_ == DT_I8) ? 1 : 0, mkind_ == MT_COS ? 1 : 0, nullptr, nullptr};
        last_batch_coarse_ = true;
        last_batch_path_ = 2;
        c.d_last_ok = nullptr;
        c.last_ok_n = 0;
        const CoarsePlan cp = plan_coarse(v, nq, dkind, ke);
        // 16-bit corpora: the fixed-bound scheme of the fp32 route without the error term — the GEMM result IS the distance, so
        // T = the k-th smallest slice minimum of the sample pass bounds the k-th best distance from above and the main pass
        // keeps every row with d <= T (no running thresholds, no compaction); a list that runs full sends the query to the
        // adaptive kernel.  (int8 distances are small integers with massive ties: they stay on the adaptive lists.)
        const CoarsePlan probe = plan_coarse(v, nq, dkind, ke, 0, 1, 1);
        if (is16 && probe.mode == 1 && coarse_fixed_enabled()) {
            double f = (double)ke / (64.0 * probe.grid_x); // aim at 64 of the 256 slots per (query, row range)
            f = std::min(0.25, std::max(0.01, f));
            // small corpora: the sample must still hold a few times k slice minima (4 per visited tile)
            const uint32_t stride = (uint32_t)std::max(1.0, std::min(std::floor(1.0 / f), std::floor(probe.tiles / (2.0 * ke))));
            const CoarsePlan cps = plan_coarse(v, nq, dkind, ke, 0, stride, 2);
            const bool tier2 = coarse_tier2_enabled();
            const size_t nM = (size_t)nq * probe.grid_x * probe.keep, nS = (size_t)nq * cps.grid_x * cps.keep, nO = (size_t)nq * ke;
            const size_t nA2 = tier2 ? (size_t)nq * cp.grid_x * cp.keep : 0;
            const size_t scratch = std::max(std::max(probe.scratch_elems, cps.scratch_elems), tier2 ? cp.scratch_elems : 0);
            const size_t qcopy = tier2 ? ((size_t)nq * qpitch + 7) / 8 : 0, flag_elems = (nq + 1) / 2 + 1;
            if (!c.need_cand(nM + nS + nA2 + nO + scratch + qcopy + 5 * flag_elems + 16) || !c.need_out(nO)) return false;
            uint64_t *cand_m = c.d_cand, *cand_s = cand_m + nM, *cand_t2 = cand_s + nS, *out2 = cand_t2 + nA2, *list_scratch = out2 + nO;
            uint64_t *q_t2 = list_scratch + scratch, *tail = q_t2 + qcopy;
            uint32_t *d_ok = reinterpret_cast<uint32_t *>(tail), *d_idx = reinterpret_cast<uint32_t *>(tail + flag_elems);
            uint32_t *d_n2 = reinterpret_cast<uint32_t *>(tail + 2 * flag_elems), *d_ovf = reinterpret_cast<uint32_t *>(tail + 4 * flag_elems);
            float *d_thr = reinterpret_cast<float *>(tail + 3 * flag_elems);
            c.d_last_ok = d_ok;
            c.last_ok_n = nq;
            bool ok = launch_coarse(ops, v.n_rows, v.dim, nq, cps, cand_s, list_scratch, st) == cudaSuccess;
            ok = ok && launch_threshold(cand_s, nq, cps.grid_x, cps.keep, ke, 0.0f, nullptr, 0.0f, (uint32_t)dim_, 0, d_thr, d_ovf, st) == cudaSuccess;
            cudaEventRecord(c.ev_start, st);
            ok = ok && launch_coarse(ops, v.n_rows, v.dim, nq, probe, cand_m, list_scratch, st, nullptr, d_thr, d_ovf) == cudaSuccess;
            cudaEventRecord(c.ev_stop, st);
            ok = ok && launch_final_select(cand_m, nq, (uint32_t)(probe.grid_x * probe.keep), ke, c.d_out, st, &lc) == cudaSuccess;
            ok = ok && launch_flags_from_overflow(d_ovf, nq, d_ok, st) == cudaSuccess;
            lc.launches += 4;
            if (tier2) {
                ok = ok && launch_compact_unproven(d_ok, nq, d_idx, d_n2, st) == cudaSuccess;
                ok = ok && launch_gather_queries(d_q, qpitch, nullptr, d_idx, d_n2, nq, q_t2, nullptr, st) == cudaSuccess;
                CoarseOperands ops2 = ops;
                ops2.queries = q_t2;
                ok = ok && launch_coarse(ops2, v.n_rows, v.dim, nq, cp, cand_t2, list_scratch, st, d_n2) == cudaSuccess;
                ok = ok && launch_final_select(cand_t2, nq, (uint32_t)(cp.grid_x * cp.keep), ke, out2, st, &lc, d_n2) == cudaSuccess;
                ok = ok && launch_scatter_rows(out2, d_idx, d_n2, nq, ke, c.d_out, d_ok, st) == cudaSuccess;
                lc.launches += 4;
            }
            coarse_batches_++;
            *d_result = c.d_out;
            return ok;
        }
        const size_t nA = (size_t)nq * cp.grid_x * cp.keep;
        if (!c.need_cand(nA + cp.scratch_elems) || !c.need_out((size_t)nq * ke)) return false;
        cudaEventRecord(c.ev_start, st);
        bool ok = launch_coarse(ops, v.n_rows, v.dim, nq, cp, c.d_cand, c.d_cand + nA, st) == cudaSuccess;
        cudaEventRecord(c.ev_stop, st);
        ok = ok && launch_final_select(c.d_cand, nq, (uint32_t)(cp.grid_x * cp.keep), ke, c.d_out, st, &lc) == cudaSuccess;
        lc.launches++;
        coarse_batches_++;
        *d_result = c.d_out;
        return ok;
    }
    CoarseKind kind = cmode == 2 ? CoarseTF32 : CoarseF16;
    // cosine: unit vectors, constant error bound, either operand kind.  L2 / raw inner product (fp32): the fp16 route only,
    // error bound from the row and query norms
    const bool unit = unit_rows();
    const bool eligible = cmode != 0 && !multi_ && !coarse_disabled_ && dtype_ == DT_F32 && (unit || cmode == 1) &&
                          (nq >= 16 || single_query_takes_coarse(ke));
    bool coarse = eligible && coarse_supported(v, nq, ke, kind);
    if (eligible && kind == CoarseF16 && (!coarse || !ensure_shadow(st))) { // rows too wide for TMEM, or no HBM for the shadow
        kind = CoarseTF32;
        coarse = unit && coarse_supported(v, nq, ke, kind);
    }
    if (coarse && !unit && !(shadow_max_abs_ <= 60000.0f)) {
        // values outside the fp16 range (or NaN): this index stays on the exact scan; give the shadow's HBM back
        coarse = false;
        std::lock_guard<std::mutex> g(mu_);
        coarse_disabled_ = true;
        cudaFree(d_shadow_);
        cudaFree(d_norm2_);
        d_shadow_ = nullptr;
        d_norm2_ = nullptr;
        shadow_cap_ = shadow_rows_ = 0;
        shadow_dirty_.clear();
    }
    last_batch_coarse_ = coarse;
    last_batch_path_ = coarse ? 1 : 0;
    if (!coarse) {
        if (!c.need_cand(sp.cand_elems) || !c.need_out((size_t)nq * ke)) return false;
        cudaEventRecord(c.ev_start, st);
        bool ok = launch_scan_topk(v, d_q, qpitch, nq, ke, sp, c.d_cand, st, &lc, nullptr, c.d_abort) == cudaSuccess;
        cudaEventRecord(c.ev_stop, st);
        ok = ok && launch_final_select(c.d_cand, nq, sp.lists_per_query * ke, ke, c.d_out, st, &lc) == cudaSuccess;
        *d_result = c.d_out;
        return ok;
    }
    // fp16 route, first tier in two passes over the shadow rows:
    //   sample pass   every `stride`-th row tile, per (query, row range) the smallest approximate distance of 8 interleaved
    //                 slices -> per query the bound T = (k-th smallest of its ranges x 8 minima) + 2 eps: k distinct rows
    //                 lie at or below it, so it bounds the k-th best distance from above
    //   main pass     all row tiles, every row with approximate distance < T is kept (fixed bound: no running thresholds,
    //                 no list compaction — ncu had the epilogue warps busy 62 % of the pass with exactly that)
    // TF32 route: one pass with adaptive lists, as before.
    const bool two_pass = kind == CoarseF16 && coarse_fixed_enabled();
    CoarsePlan cp = plan_coarse(v, nq, kind, ke); // TF32 / single-pass: the adaptive lists ARE the first tier
    CoarsePlan cps{};                             // sample pass
    if (two_pass) {
        // expected rows below T per (query, row range) = k / (sample fraction * ranges): aim at 24 of the 96 slots
        const CoarsePlan probe = plan_coarse(v, nq, kind, ke, 0, 1, 1);
        double f = (double)ke / (24.0 * probe.grid_x);
        f = std::min(0.25, std::max(0.01, f));
        // small corpora: the sample must still hold a few times k slice minima (4 per visited tile)
        const uint32_t stride = (uint32_t)std::max(1.0, std::min(std::floor(1.0 / f), std::floor(probe.tiles / (2.0 * ke))));
        cps = plan_coarse(v, nq, kind, ke, 0, stride, 2);
        cp = probe;
    }
    const size_t per_query = (size_t)cp.grid_x * cp.keep;
    // second tier (fp16 route): the queries whose first-tier proof failed (a list of the main pass overflowed: more than 96
    // rows of one range within the bound — clustered corpora) are packed to the front and run once more with adaptive
    // lists of 128 per row range.  Nothing is known on the host: the tier's kernels read the count of open queries from
    // device memory and leave at once when it is zero.
    const bool tier2 = kind == CoarseF16 && coarse_tier2_enabled();
    CoarsePlan cp2{};
    if (tier2) cp2 = plan_coarse(v, nq, kind, ke, kCoarseKeepWide);
    const size_t nA = (size_t)nq * per_query, nO = (size_t)nq * ke;
    const size_t nS = two_pass ? (size_t)nq * cps.grid_x * cps.keep : 0;
    const size_t nA2 = tier2 ? (size_t)nq * cp2.grid_x * cp2.keep : 0;
    const size_t q16_pitch = (dim_ * 2 + 15) & ~(size_t)15;
    const size_t q16_elems = kind == CoarseF16 ? ((size_t)nq * q16_pitch + 7) / 8 : 0;
    const size_t qn_elems = unit ? 0 : (nq + 1) / 2 + 1; // |q|^2 per query (floats)
    const size_t scratch = std::max(std::max(cp.scratch_elems, two_pass ? cps.scratch_elems : 0), tier2 ? cp2.scratch_elems : 0);
    const size_t flag_elems = (nq + 1) / 2 + 1; // nq uint32 / float values
    const size_t total = nA + nS + nA2 + 2 * nO + sp.cand_elems + (tier2 ? 2 : 1) * (q16_elems + qn_elems) + scratch + 5 * flag_elems + 16;
    if (!c.need_cand(total) || !c.need_out(nO)) return false;
    uint64_t *coarse_cand = c.d_cand, *cand_s = coarse_cand + nA, *cand_t2 = cand_s + nS, *out1 = cand_t2 + nA2, *out2 = out1 + nO,
             *cand2 = out2 + nO;
    uint64_t *q16 = cand2 + sp.cand_elems;
    uint64_t *q16_t2 = q16 + q16_elems;
    uint64_t *list_scratch = q16_t2 + (tier2 ? q16_elems : 0);
    uint64_t *tail = list_scratch + scratch;
    float *d_qn2 = unit ? nullptr : reinterpret_cast<float *>(tail);
    float *d_qn2_t2 = (unit || !tier2) ? nullptr : reinterpret_cast<float *>(tail + qn_elems);
    tail += (tier2 ? 2 : 1) * qn_elems;
    uint32_t *d_ok = reinterpret_cast<uint32_t *>(tail);
    uint32_t *d_idx = reinterpret_cast<uint32_t *>(tail + flag_elems); // tier 2: indices of the open queries
    uint32_t *d_n2 = reinterpret_cast<uint32_t *>(tail + 2 * flag_elems); //         and their count
    float *d_thr = reinterpret_cast<float *>(tail + 3 * flag_elems);       // fixed bound per query
    uint32_t *d_ovf = reinterpret_cast<uint32_t *>(tail + 4 * flag_elems); // a list of the main pass ran full
    c.d_last_ok = d_ok;
    c.last_ok_n = nq;
    CoarseOperands ops{v.rows, v.pitch, d_q, qpitch, 0, 0, nullptr, nullptr};
    bool ok = true;
    if (kind == CoarseF16) {
        ok = launch_to_f16(d_q, qpitch, (uint32_t)dim_, 0, nq, q16, q16_pitch, st) == cudaSuccess;
        ops = CoarseOperands{d_shadow_, 0, q16, q16_pitch, 0, mkind_ == MT_L2 ? 1 : 0, d_norm2_, d_qn2};
        if (!unit) ok = ok && launch_row_stats(d_q, qpitch, (uint32_t)dim_, 0, nq, d_qn2, nullptr, st) == cudaSuccess;
        lc.launches += unit ? 1 : 2;
    }
    const float eps = coarse_eps(kind);
    if (two_pass) {
        ok = ok && launch_coarse(ops, v.n_rows, v.dim, nq, cps, cand_s, list_scratch, st) == cudaSuccess;
        ok = ok && launch_threshold(cand_s, nq, cps.grid_x, cps.keep, ke, eps, d_qn2, shadow_max_norm_, (uint32_t)dim_, mkind_ == MT_L2 ? 1 : 0, d_thr,
                                    d_ovf, st) == cudaSuccess;
        lc.launches += 2;
    }
    cudaEventRecord(c.ev_start, st);
    ok = ok && launch_coarse(ops, v.n_rows, v.dim, nq, cp, coarse_cand, list_scratch, st, nullptr, two_pass ? d_thr : nullptr,
                             two_pass ? d_ovf : nullptr) == cudaSuccess;
    cudaEventRecord(c.ev_stop, st);
    // exact rescoring of the few candidates that can still matter + exact top-k + proof, one CTA per query
    ok = ok && launch_refine(v, d_q, qpitch, nq, cp.grid_x, cp.keep, ke, coarse_cand, eps, d_qn2, shadow_max_norm_, d_ok, out1, nullptr, nullptr,
                             st, two_pass ? d_thr : nullptr, two_pass ? d_ovf : nullptr) == cudaSuccess;
    lc.launches += 2;
    if (tier2) {
        ok = ok && launch_compact_unproven(d_ok, nq, d_idx, d_n2, st) == cudaSuccess;
        ok = ok && launch_gather_queries(q16, q16_pitch, d_qn2, d_idx, d_n2, nq, q16_t2, d_qn2_t2, st) == cudaSuccess;
        CoarseOperands ops2 = ops;
        ops2.queries = q16_t2;
        ops2.q_norm2 = d_qn2_t2;
        ok = ok && launch_coarse(ops2, v.n_rows, v.dim, nq, cp2, cand_t2, list_scratch, st, d_n2) == cudaSuccess;
        ok = ok && launch_refine(v, d_q, qpitch, nq, cp2.grid_x, cp2.keep, ke, cand_t2, eps, d_qn2_t2, shadow_max_norm_, d_ok, out1, d_idx, d_n2,
                                 st) == cudaSuccess;
        lc.launches += 4;
    }
    // exact fallback, entirely on device: CTAs whose queries are all verified exit at once
    ok = ok && launch_scan_topk(v, d_q, qpitch, nq, ke, sp, cand2, st, &lc, d_ok, c.d_abort) == cudaSuccess;
    ok = ok && launch_final_select(cand2, nq, sp.lists_per_query * ke, ke, out2, st, &lc) == cudaSuccess;
    ok = ok && launch_blend(d_ok, out1, out2, nq, ke, c.d_out, st, &lc) == cudaSuccess;
    coarse_batches_++;
    *d_result = c.d_out;
    return ok;
}

int FlatIndex::topk_batch(const void *qs, size_t qstride, size_t nq, size_t k, VecSimQueryParams *qp, size_t *out_labels,
                          double *out_scores) {
    void *tctx = qp ? qp->timeoutCtx : nullptr;
    last_mode_ = STANDARD_KNN;
    const double nan = std::numeric_limits<double>::quiet_NaN();
    for (size_t i = 0; i < nq * k; i++) {
        out_labels[i] = SIZE_MAX;
        out_scores[i] = nan;
    }
    if (nq == 0 || k == 0) return VecSim_QueryReply_OK;
    if (!flush()) return -1;
    const size_t n = count_;
    if (n == 0) return VecSim_QueryReply_OK;
    if (timed_out(tctx)) return VecSim_QueryReply_TimedOut;
    if (multi_ || std::min(k, n) > (size_t)kMaxFusedK) { // generic path, one query at a time
        for (size_t i = 0; i < nq; i++) {
            VecSimQueryReply *r = topk(static_cast<const uint8_t *>(qs) + i * qstride, k, qp, BY_SCORE);
            const int code = r->code;
            for (size_t j = 0; j < r->results.size() && j < k; j++) {
                out_labels[i * k + j] = r->results[j].id;
                out_scores[i * k + j] = r->results[j].score;
            }
            delete r;
            if (code != VecSim_QueryReply_OK) return code;
        }
        return VecSim_QueryReply_OK;
    }
    auto c = checkout();
    if (!c) return -1;
    const size_t qpitch = (stored_bytes_ + 15) & ~(size_t)15;
    const uint32_t ke = (uint32_t)std::min(k, n);
    const CorpusView v = view();
    LaunchCounters lc;
    bool ok = c->need_query(qpitch * nq);
    if (ok) {
        memset(c->h_query, 0, qpitch * nq);
        for (size_t i = 0; i < nq; i++) preprocess_query(static_cast<const uint8_t *>(qs) + i * qstride, c->h_query + i * qpitch);
        ok = cudaMemcpyAsync(c->d_query, c->h_query, qpitch * nq, cudaMemcpyHostToDevice, c->stream) == cudaSuccess;
    }
    uint64_t *d_res = nullptr;
    ok = ok && batch_scan(*c, c->d_query, qpitch, (uint32_t)nq, ke, c->stream, lc, &d_res);
    ok = ok && cudaMemcpyAsync(c->h_out, c->d_out, nq * ke * 8, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess;
    launches_total_ += lc.launches;
    if (ok) {
        const int w = wait_polling(c->stream, tctx); // a 414 ms exact-scan fallback no longer holds a timed-out caller
        if (w == 1) {
            c->abandoned = true;
                *c->h_abort = 1; // the kernels still running on its stream wind down
            checkin(std::move(c));
            return VecSim_QueryReply_TimedOut;
        }
        ok = w == 0;
    }
    if (ok) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, c->ev_start, c->ev_stop) == cudaSuccess) {
            std::lock_guard<std::mutex> g(stats_mu_);
            scan_us_ += ms * 1000.0;
            scan_launches_++;
            scan_bytes_ += (uint64_t)n * stored_bytes_;
        }
        std::vector<VecSimQueryResult> tmp;
        VecSimQueryReply rr;
        for (size_t i = 0; i < nq; i++) {
            rr.results.clear();
            for (uint32_t j = 0; j < ke; j++) {
                const uint64_t comp = c->h_out[i * ke + j];
                if (comp == kEmptySlot) break;
                rr.results.push_back({id_to_label_[(uint32_t)comp], (double)key_to_float((uint32_t)(comp >> 32))});
            }
            finish_reply(&rr, BY_SCORE);
            for (size_t j = 0; j < rr.results.size(); j++) {
                out_labels[i * k + j] = rr.results[j].id;
                out_scores[i * k + j] = rr.results[j].score;
            }
        }
    }
    checkin(std::move(c));
    if (!ok) return -1;
    if (timed_out(tctx)) return VecSim_QueryReply_TimedOut;
    return VecSim_QueryReply_OK;
}

int FlatIndex::topk_batch_device(const void *d_q, size_t nq, size_t k, int64_t *d_labels, float *d_scores, cudaStream_t s) {
    if (nq == 0 || k == 0) return 0;
    if (!flush() || !sync_labels_to_device()) return -1;
    const size_t n = count_;
    if (multi_ || k > (size_t)kMaxFusedK) return -1;
    // Scratch of this entry point is stream-ordered: one dedicated context, reused call after call.
    // Callers enqueue on one stream (or synchronise between streams), as with any async API.
    std::lock_guard<std::mutex> dg(dev_mu_);
    if (!dev_ctx_) dev_ctx_ = checkout();
    QueryCtx *c = dev_ctx_.get();
    if (!c) return -1;
    collect_dev_timing_locked(); // the previous call's scan events (stream-ordered before this call)
    const size_t qpitch = (stored_bytes_ + 15) & ~(size_t)15;
    const uint32_t ke = (uint32_t)std::min(k, std::max<size_t>(n, 1));
    cudaStream_t st = s ? s : cudaStreamLegacy; // NULL = the legacy default stream, as everywhere in CUDA
    LaunchCounters lc;
    bool ok = true;
    if (n == 0) {
        ok = cudaMemsetAsync(d_labels, 0xFF, nq * k * 8, st) == cudaSuccess;
    } else {
        uint64_t *d_res = nullptr;
        ok = c->need_out(nq * k);
        if (!ok) {
        } else if (ke == k) {
            ok = batch_scan(*c, d_q, qpitch, (uint32_t)nq, ke, st, lc, &d_res);
        } else {
            // fewer rows than k: select [nq][ke], then widen the rows to [nq][k] (tail = empty)
            ok = batch_scan(*c, d_q, qpitch, (uint32_t)nq, ke, st, lc, &d_res);
            ok = ok && c->need_ids(nq * k * 2);
            uint64_t *wide = reinterpret_cast<uint64_t *>(c->d_ids);
            ok = ok && cudaMemsetAsync(wide, 0xFF, nq * k * 8, st) == cudaSuccess;
            ok = ok && cudaMemcpy2DAsync(wide, k * 8, d_res, ke * 8, ke * 8, nq, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
            ok = ok && cudaMemcpyAsync(c->d_out, wide, nq * k * 8, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
        }
        ok = ok && launch_unpack_results(c->d_out, (uint32_t)nq, (uint32_t)k, d_id_to_label_, d_labels, d_scores, st, &lc) == cudaSuccess;
        dev_timing_pending_ = ok;
        dev_timing_bytes_ = (uint64_t)n * stored_bytes_;
    }
    launches_total_ += lc.launches;
    return ok ? 0 : -1;
}

VecSimQueryReply *FlatIndex::range(const void *q, double radius, VecSimQueryParams *qp, VecSimQueryReply_Order order) {
    auto *rep = new VecSimQueryReply();
    last_mode_ = RANGE_QUERY;
    void *tctx = qp ? qp->timeoutCtx : nullptr;
    if (!flush()) return rep;
    const size_t n = count_;
    if (n == 0) return rep;
    if (timed_out(tctx)) {
        rep->code = VecSim_QueryReply_TimedOut;
        return rep;
    }
    auto c = checkout();
    if (!c) return rep;
    const size_t qpitch = (stored_bytes_ + 15) & ~(size_t)15;
    LaunchCounters lc;
    bool ok = c->need_query(qpitch) && c->need_scores(n) && c->need_cand(n);
    if (ok) {
        memset(c->h_query, 0, qpitch);
        preprocess_query(q, c->h_query);
        ok = upload_query(*c, c->h_query, 1);
    }
    const CorpusView v = view();
    ok = ok && launch_scan_scores(v, c->d_query, c->d_scores, c->stream, &lc) == cudaSuccess;
    ok = ok && launch_range_compact(c->d_scores, (uint32_t)n, (float)radius, c->d_cand, c->d_count, c->stream, &lc) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(c->h_count, c->d_count, 4, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(c->stream) == cudaSuccess;
    if (ok) {
        const uint32_t m = *c->h_count;
        ok = c->need_out(m);
        ok = ok && cudaMemcpyAsync(c->h_out, c->d_cand, (size_t)m * 8, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess;
        ok = ok && cudaStreamSynchronize(c->stream) == cudaSuccess;
        if (ok) {
            if (multi_) { // best score per label (brute_force_multi.h range container)
                std::unordered_map<size_t, uint32_t> best;
                for (uint32_t i = 0; i < m; i++) {
                    const uint64_t comp = c->h_out[i];
                    const size_t label = id_to_label_[(uint32_t)comp];
                    const uint32_t key = (uint32_t)(comp >> 32);
                    auto it = best.find(label);
                    if (it == best.end() || key < it->second) best[label] = key;
                }
                for (auto &kv : best) rep->results.push_back({kv.first, (double)key_to_float(kv.second)});
            } else {
                rep->results.reserve(m);
                for (uint32_t i = 0; i < m; i++) {
                    const uint64_t comp = c->h_out[i];
                    rep->results.push_back({id_to_label_[(uint32_t)comp], (double)key_to_float((uint32_t)(comp >> 32))});
                }
            }
        }
    }
    launches_total_ += lc.launches;
    checkin(std::move(c));
    if (!ok) rep->results.clear();
    if (timed_out(tctx)) rep->code = VecSim_QueryReply_TimedOut; // brute_force.h:306-309 keeps partial results
    finish_reply(rep, order);
    return rep;
}

double FlatIndex::distance_from(size_t label, const void *blob) {
    const double nan = std::numeric_limits<double>::quiet_NaN();
    std::vector<idType> ids;
    {
        std::lock_guard<std::mutex> g(mu_);
        if (multi_) {
            auto it = label_to_ids_.find(label);
            if (it == label_to_ids_.end()) return nan;
            ids = it->second;
        } else {
            auto it = label_to_id_.find(label);
            if (it == label_to_id_.end()) return nan;
            ids.push_back(it->second);
        }
    }
    if (!flush()) return nan;
    auto c = checkout();
    if (!c) return nan;
    LaunchCounters lc;
    bool ok = c->need_ids(ids.size()) && upload_query(*c, static_cast<const uint8_t *>(blob), 1);
    if (ok) {
        for (size_t i = 0; i < ids.size(); i++) c->h_ids[i] = ids[i];
        ok = cudaMemcpyAsync(c->d_ids, c->h_ids, ids.size() * 4, cudaMemcpyHostToDevice, c->stream) == cudaSuccess;
    }
    ok = ok && launch_gather_distances(view(), c->d_query, c->d_ids, (uint32_t)ids.size(), c->d_dist, c->stream, &lc) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(c->h_dist, c->d_dist, ids.size() * 4, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(c->stream) == cudaSuccess;
    double best = nan;
    if (ok) { // brute_force_multi.h:234-238: the min over the label's rows, folded in their order as `(dist < d) ? dist : d`,
              // so a NaN row is replaced by the next row and the answer is NaN only when the last row is NaN
        float dist = std::numeric_limits<float>::infinity();
        for (size_t i = 0; i < ids.size(); i++) dist = (dist < c->h_dist[i]) ? dist : c->h_dist[i];
        best = (double)dist;
    }
    launches_total_ += lc.launches;
    checkin(std::move(c));
    return best;
}

// brute_force.h:380-451, thresholds and float/double comparison types reproduced exactly.
bool FlatIndex::prefer_adhoc(size_t subset, size_t k, bool initial) {
    (void)k;
    const size_t index_size = count_;
    subset = std::min(subset, index_size);
    const size_t d = dim_;
    const float r = (index_size == 0) ? 0.0f : (float)subset / (float)label_count();
    bool res;
    if (index_size <= 5500) {
        res = true;
    } else if (d <= 300) {
        if (r <= 0.15)
            res = true;
        else if (r <= 0.35)
            res = (d <= 75) ? false : (index_size <= 550000);
        else
            res = false;
    } else {
        if (r <= 0.55)
            res = true;
        else if (d <= 750)
            res = false;
        else
            res = (r <= 0.75);
    }
    last_mode_ = res ? (initial ? HYBRID_ADHOC_BF : HYBRID_BATCHES_TO_ADHOC_BF) : HYBRID_BATCHES;
    return res;
}

// ------------------------------------------------------------------------------------------------
// batch iterator
// ------------------------------------------------------------------------------------------------
BatchIter *FlatIndex::batch_new(const void *q, VecSimQueryParams *qp) {
    auto *it = new BatchIter();
    it->index = this;
    it->query.assign((stored_bytes_ + 15) & ~(size_t)15, 0);
    preprocess_query(q, it->query.data()); // forced copy, brute_force.h:371-372
    it->timeout_ctx = qp ? qp->timeoutCtx : nullptr;
    it->label_count = label_count();
    return it;
}

VecSimQueryReply *FlatIndex::batch_next(BatchIter *it, size_t n_res, VecSimQueryReply_Order order) {
    auto *rep = new VecSimQueryReply();
    if (!it->scored) {
        // first call: the only time the index is read (bf_batch_iterator.h:176-189)
        if (!flush()) return rep;
        it->n_rows = (uint32_t)count_;
        it->label_count = label_count();
        it->id_to_label_snap = id_to_label_;
        if (timed_out(it->timeout_ctx)) {
            rep->code = VecSim_QueryReply_TimedOut;
            return rep;
        }
        if (!it->ctx) it->ctx = checkout();
        if (!it->ctx) return rep;
        if (it->n_rows) {
            LaunchCounters lc;
            bool ok = it->ctx->need_scores(it->n_rows) && upload_query(*it->ctx, it->query.data(), 1);
            // upload_query copies stored_bytes_ from a tightly packed source
            ok = ok && launch_scan_scores(view(), it->ctx->d_query, it->ctx->d_scores, it->ctx->stream, &lc) == cudaSuccess;
            ok = ok && cudaStreamSynchronize(it->ctx->stream) == cudaSuccess;
            launches_total_ += lc.launches;
            {
                std::lock_guard<std::mutex> g(stats_mu_);
                scan_launches_++;
                scan_bytes_ += (uint64_t)it->n_rows * stored_bytes_;
            }
            if (!ok) return rep;
        }
        it->scored = true;
    }
    if (timed_out(it->timeout_ctx)) {
        rep->code = VecSim_QueryReply_TimedOut;
        return rep;
    }
    const size_t remaining_labels = it->label_count - it->returned;
    const size_t want_labels = std::min(n_res, remaining_labels);
    size_t produced = 0;
    while (produced < want_labels) {
        const size_t want = multi_ ? std::max<size_t>(2 * (want_labels - produced), 64) : (want_labels - produced);
        const long got = select_from_scores(*it->ctx, it->n_rows, it->has_cursor, it->cursor, std::min<size_t>(want, it->n_rows));
        if (got <= 0) break;
        for (long i = 0; i < got; i++) {
            const uint64_t comp = it->ctx->h_out[i];
            if (produced < want_labels) {
                const size_t label = it->id_to_label_snap[(uint32_t)comp];
                it->has_cursor = true;
                it->cursor = comp;
                if (multi_ && !it->seen.insert(label).second) continue;
                rep->results.push_back({label, (double)key_to_float((uint32_t)(comp >> 32))});
                produced++;
            } else {
                break; // leave the rest for the next call: cursor stays on the last consumed entry
            }
        }
        if ((size_t)got < std::min<size_t>(want, it->n_rows)) break;
    }
    it->returned += rep->results.size();
    finish_reply(rep, order == BY_ID ? BY_ID : BY_SCORE);
    return rep;
}

// ------------------------------------------------------------------------------------------------
// ad-hoc context
// ------------------------------------------------------------------------------------------------
AdhocCtx *FlatIndex::adhoc_new(const void *q) {
    auto *a = new AdhocCtx();
    a->index = this;
    a->query.assign(stored_bytes_, 0);
    preprocess_query(q, a->query.data()); // the context normalises internally (hybrid_reader.c:212-214)
    a->ctx = checkout();
    if (!a->ctx) {
        delete a;
        return nullptr;
    }
    return a;
}

void FlatIndex::adhoc_distances(AdhocCtx *a, const size_t *labels, double *out, size_t n) {
    const double nan = std::numeric_limits<double>::quiet_NaN();
    for (size_t i = 0; i < n; i++) out[i] = nan;
    if (n == 0 || !flush()) return;
    QueryCtx &c = *a->ctx;
    LaunchCounters lc;
    // expand labels to row ids (multi: several rows per label, min taken on the host)
    std::vector<uint32_t> ids;
    std::vector<uint32_t> owner;
    ids.reserve(n);
    {
        std::lock_guard<std::mutex> g(mu_);
        for (size_t i = 0; i < n; i++) {
            if (multi_) {
                auto it = label_to_ids_.find(labels[i]);
                if (it == label_to_ids_.end()) continue;
                for (idType id : it->second) {
                    ids.push_back(id);
                    owner.push_back((uint32_t)i);
                }
            } else {
                auto it = label_to_id_.find(labels[i]);
                if (it == label_to_id_.end()) continue;
                ids.push_back(it->second);
                owner.push_back((uint32_t)i);
            }
        }
    }
    if (ids.empty()) return;
    bool ok = c.need_ids(ids.size());
    if (ok && !a->query_on_device) {
        ok = upload_query(c, a->query.data(), 1);
        a->query_on_device = ok;
    }
    if (ok) {
        memcpy(c.h_ids, ids.data(), ids.size() * 4);
        ok = cudaMemcpyAsync(c.d_ids, c.h_ids, ids.size() * 4, cudaMemcpyHostToDevice, c.stream) == cudaSuccess;
    }
    ok = ok && launch_gather_distances(view(), c.d_query, c.d_ids, (uint32_t)ids.size(), c.d_dist, c.stream, &lc) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(c.h_dist, c.d_dist, ids.size() * 4, cudaMemcpyDeviceToHost, c.stream) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(c.stream) == cudaSuccess;
    launches_total_ += lc.launches;
    if (!ok) return;
    // the same fold as distance_from over each label's rows in their order (brute_force_multi.h:234-238)
    std::vector<float> dist(n, std::numeric_limits<float>::infinity());
    for (size_t i = 0; i < ids.size(); i++) {
        float &d = dist[owner[i]];
        d = (d < c.h_dist[i]) ? d : c.h_dist[i];
    }
    for (size_t i = 0; i < ids.size(); i++) out[owner[i]] = (double)dist[owner[i]];
}


// ------------------------------------------------------------------------------------------------
// fused hybrid ad-hoc query (HybridIterator in HYBRID_ADHOC_BF mode, src/iterators/hybrid_reader.c:289-335:
// child docIds in ascending order -> GetDistanceFrom each -> heap of the k best, strict `<` admission, NaN = deleted)
// ------------------------------------------------------------------------------------------------
bool FlatIndex::sync_label_table() {
    std::lock_guard<std::mutex> g(mu_);
    if (!l2i_dirty_ && d_label_to_id_) return true;
    size_t max_label = 0;
    for (size_t i = 0; i < count_; i++) max_label = std::max(max_label, id_to_label_[i]);
    if (max_label > 4 * count_ + (1u << 24) || max_label >= 0xFFFFFFFFull) return false; // sparse labels: no dense table
    const size_t size = max_label + 1;
    std::vector<uint32_t> tab(size, 0xFFFFFFFFu);
    for (size_t i = 0; i < count_; i++) tab[id_to_label_[i]] = (uint32_t)i;
    if (size > l2i_cap_) {
        cudaFree(d_label_to_id_);
        d_label_to_id_ = nullptr;
        const size_t cap = size + size / 4 + 1024;
        CU_OK(cudaMalloc(&d_label_to_id_, cap * 4));
        l2i_cap_ = cap;
    }
    CU_OK(cudaMemcpy(d_label_to_id_, tab.data(), size * 4, cudaMemcpyHostToDevice));
    l2i_size_ = size;
    l2i_dirty_ = false;
    return true;
}

int FlatIndex::topk_filtered(const void *q, size_t k, const uint32_t *doc_ids, size_t n, bool ids_on_device, size_t *out_labels,
                             double *out_scores, size_t *out_count) {
    *out_count = 0;
    last_mode_ = HYBRID_ADHOC_BF;
    if (k == 0 || n == 0) return 0;
    if (multi_ || n > 0xFFFFFFF0ull) return -2;
    if (!flush()) return -1;
    if (count_ == 0) return 0;
    if (!sync_label_table()) return -2;
    auto c = checkout();
    if (!c) return -1;
    const size_t qpitch = (stored_bytes_ + 15) & ~(size_t)15;
    LaunchCounters lc;
    bool ok = c->need_query(qpitch) && c->need_ids(2 * n + 256) && c->need_scores(n);
    if (ok) {
        memset(c->h_query, 0, qpitch);
        preprocess_query(q, c->h_query);
        ok = upload_query(*c, c->h_query, 1);
    }
    // d_ids: [0,n) row ids, [n,2n) the labels when they arrive from the host
    const uint32_t *d_labels = doc_ids;
    if (ok && !ids_on_device) {
        ok = cudaMemcpyAsync(c->d_ids + n, doc_ids, n * 4, cudaMemcpyHostToDevice, c->stream) == cudaSuccess;
        d_labels = c->d_ids + n;
    }
    ok = ok && launch_map_labels(d_labels, (uint32_t)n, d_label_to_id_, (uint32_t)l2i_size_, c->d_ids, c->stream, &lc) == cudaSuccess;
    ok = ok && launch_gather_distances(view(), c->d_query, c->d_ids, (uint32_t)n, c->d_scores, c->stream, &lc) == cudaSuccess;
    launches_total_ += lc.launches;
    if (!ok) {
        checkin(std::move(c));
        return -1;
    }
    // k best positions by (distance asc, position asc) = (distance, docId): NaN (deleted docs) sort last and are dropped
    const size_t want = std::min(k, n);
    const long got = select_from_scores(*c, (uint32_t)n, false, 0, want);
    if (got < 0) {
        checkin(std::move(c));
        return -1;
    }
    LaunchCounters lc2;
    uint32_t *d_sel = c->d_ids; // row ids are no longer needed
    ok = launch_pick_labels(c->d_out, (uint32_t)got, d_labels, d_sel, c->stream, &lc2) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(c->h_ids, d_sel, (size_t)got * 4, cudaMemcpyDeviceToHost, c->stream) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(c->stream) == cudaSuccess;
    launches_total_ += lc2.launches;
    size_t w = 0;
    if (ok)
        for (long i = 0; i < got; i++) {
            const float d = key_to_float((uint32_t)(c->h_out[i] >> 32));
            if (std::isnan(d)) continue;
            out_labels[w] = c->h_ids[i];
            out_scores[w] = (double)d;
            w++;
        }
    *out_count = w;
    checkin(std::move(c));
    return ok ? 0 : -1;
}


// The same for MANY queries (BASELINE configs[4]: a batch of hybrid queries, each with its own filter set): every query's chain
// (labels -> rows, gathered distances, selection, label pick, D2H) is enqueued on its own context's stream before anything is
// waited for, so the chains overlap and the host pays one round of synchronisations instead of two per query.  Device-resident
// id lists only (the filters' AND / OR results).
int FlatIndex::topk_filtered_batch(const void *const *queries, size_t nq, size_t k, const uint32_t *const *d_doc_ids, const size_t *counts,
                                   size_t *out_labels, double *out_scores, size_t *out_counts) {
    for (size_t i = 0; i < nq; i++) out_counts[i] = 0;
    last_mode_ = HYBRID_ADHOC_BF;
    if (k == 0 || nq == 0) return 0;
    if (multi_ || k > (size_t)kMaxFusedK) return -2;
    if (!flush()) return -1;
    if (count_ == 0) return 0;
    if (!sync_label_table()) return -2;
    const size_t qpitch = (stored_bytes_ + 15) & ~(size_t)15;
    constexpr size_t kWave = 16; // contexts in flight at once
    int rc = 0;
    for (size_t q0 = 0; q0 < nq && rc == 0; q0 += kWave) {
        const size_t q1 = std::min(nq, q0 + kWave);
        struct Job {
            std::unique_ptr<QueryCtx> c;
            size_t want = 0;
            bool ok = false;
        };
        std::vector<Job> jobs(q1 - q0);
        LaunchCounters lc;
        for (size_t qi = q0; qi < q1; qi++) {
            Job &j = jobs[qi - q0];
            const size_t n = counts[qi];
            if (n == 0) continue;
            if (n > 0xFFFFFFF0ull) {
                rc = -2;
                break;
            }
            j.c = checkout();
            if (!j.c) {
                rc = -1;
                break;
            }
            QueryCtx &c = *j.c;
            j.want = std::min(k, n);
            const uint32_t lists = plan_select_scores_lists((uint32_t)n);
            bool ok = c.need_query(qpitch) && c.need_ids(2 * n + 256) && c.need_scores(n) && c.need_out(j.want + 1) &&
                      c.need_cand((size_t)lists * j.want);
            if (ok) {
                memset(c.h_query, 0, qpitch);
                preprocess_query(queries[qi], c.h_query);
                ok = upload_query(c, c.h_query, 1);
            }
            const uint32_t *d_labels = d_doc_ids[qi];
            ok = ok && launch_map_labels(d_labels, (uint32_t)n, d_label_to_id_, (uint32_t)l2i_size_, c.d_ids, c.stream, &lc) == cudaSuccess;
            ok = ok && launch_gather_distances(view(), c.d_query, c.d_ids, (uint32_t)n, c.d_scores, c.stream, &lc) == cudaSuccess;
            ok = ok && launch_select_scores(c.d_scores, (uint32_t)n, nullptr, (uint32_t)j.want, c.d_cand, c.stream, &lc) == cudaSuccess;
            ok = ok && launch_final_select(c.d_cand, 1, lists * (uint32_t)j.want, (uint32_t)j.want, c.d_out, c.stream, &lc) == cudaSuccess;
            ok = ok && cudaMemcpyAsync(c.h_out, c.d_out, j.want * 8, cudaMemcpyDeviceToHost, c.stream) == cudaSuccess;
            // the selected positions -> labels (empty slots pick nothing that is read back: they are cut below)
            ok = ok && launch_pick_labels(c.d_out, (uint32_t)j.want, d_labels, c.d_ids, c.stream, &lc) == cudaSuccess;
            ok = ok && cudaMemcpyAsync(c.h_ids, c.d_ids, j.want * 4, cudaMemcpyDeviceToHost, c.stream) == cudaSuccess;
            j.ok = ok;
            if (!ok) rc = -1;
        }
        launches_total_ += lc.launches;
        for (size_t qi = q0; qi < q1; qi++) { // one round of waits; contexts go back even on failure
            Job &j = jobs[qi - q0];
            if (!j.c) continue;
            const bool synced = cudaStreamSynchronize(j.c->stream) == cudaSuccess;
            if (j.ok && synced && rc == 0) {
                size_t w = 0;
                for (size_t i = 0; i < j.want; i++) {
                    if (j.c->h_out[i] == kEmptySlot) break;
                    const float d = key_to_float((uint32_t)(j.c->h_out[i] >> 32));
                    if (std::isnan(d)) continue;
                    out_labels[qi * k + w] = j.c->h_ids[i];
                    out_scores[qi * k + w] = (double)d;
                    w++;
                }
                out_counts[qi] = w;
            } else if (!synced) {
                rc = -1;
            }
            checkin(std::move(j.c));
        }
    }
    return rc;
}

// ------------------------------------------------------------------------------------------------
// request combiner for the stock single-query entry point (opt-in)
// ------------------------------------------------------------------------------------------------
struct FlatIndex::TopkReq {
    const void *blob;
    std::vector<size_t> labels;
    std::vector<double> scores;
    int code = VecSim_QueryReply_OK;
};

int FlatIndex::microbatch_window_us() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("VECSIM_B200_MICROBATCH_US");
        v = e ? std::max(0, atoi(e)) : 0;
    }
    return v;
}

VecSimQueryReply *FlatIndex::topk_combined(const void *q, size_t k, VecSimQueryParams *qp, VecSimQueryReply_Order order) {
    const int window = microbatch_window_us();
    // only what the batched entry point serves in one pass; everything else keeps the direct route
    if (window <= 0 || multi_ || k == 0 || k > (size_t)kMaxFusedK || count_ < 65536) return topk(q, k, qp, order);
    // fp16 / bf16 corpora: a combined batch >= 16 would ride the tensor-core direct route, whose scores are within the 1e-2
    // bar but not bit-identical with the single-query scan — the answer would depend on how many callers were concurrent
    if (dtype_ == DT_F16 || dtype_ == DT_BF16) return topk(q, k, qp, order);
    void *tctx = qp ? qp->timeoutCtx : nullptr;
    auto *rep = new VecSimQueryReply();
    last_mode_ = STANDARD_KNN;
    if (timed_out(tctx)) {
        rep->code = VecSim_QueryReply_TimedOut;
        return rep;
    }
    using Batcher = MicroBatcher<TopkReq>;
    std::shared_ptr<void> holder;
    {
        std::lock_guard<std::mutex> g(mb_mu_);
        auto &slot = batchers_[k];
        if (!slot) {
            const size_t blob_bytes = dim_ * elem_bytes_;
            slot = std::shared_ptr<void>(
                new Batcher(256, std::chrono::microseconds(window),
                            [this, k, blob_bytes](std::vector<TopkReq *> &reqs) {
                                const size_t nq = reqs.size();
                                std::vector<uint8_t> blobs(nq * blob_bytes);
                                for (size_t i = 0; i < nq; i++) memcpy(blobs.data() + i * blob_bytes, reqs[i]->blob, blob_bytes);
                                std::vector<size_t> labels(nq * k);
                                std::vector<double> scores(nq * k);
                                const int code = topk_batch(blobs.data(), blob_bytes, nq, k, nullptr, labels.data(), scores.data());
                                for (size_t i = 0; i < nq; i++) {
                                    reqs[i]->code = code;
                                    reqs[i]->labels.assign(labels.begin() + i * k, labels.begin() + (i + 1) * k);
                                    reqs[i]->scores.assign(scores.begin() + i * k, scores.begin() + (i + 1) * k);
                                }
                            },
                            [](TopkReq &r) { r.code = -1; }),
                [](void *p) { delete static_cast<Batcher *>(p); });
        }
        holder = slot;
    }
    TopkReq r;
    r.blob = q;
    static_cast<Batcher *>(holder.get())->submit(r);
    if (r.code == VecSim_QueryReply_TimedOut || timed_out(tctx)) {
        rep->code = VecSim_QueryReply_TimedOut;
        return rep;
    }
    if (r.code != VecSim_QueryReply_OK) {
        log("warning", "vecsim_b200: combined top-k query failed on device");
        return rep;
    }
    for (size_t j = 0; j < k && j < r.labels.size(); j++)
        if (r.labels[j] != SIZE_MAX) rep->results.push_back({r.labels[j], r.scores[j]});
    finish_reply(rep, order);
    return rep;
}

// ------------------------------------------------------------------------------------------------
// info
// ------------------------------------------------------------------------------------------------
VecSimIndexBasicInfo FlatIndex::basic_info() const {
    VecSimIndexBasicInfo i{};
    i.algo = VecSimAlgo_BF;
    i.metric = metric_;
    i.type = type_;
    i.isMulti = multi_;
    i.isTiered = false;
    i.isDisk = false;
    i.blockSize = block_size_;
    i.dim = dim_;
    return i;
}
VecSimIndexStatsInfo FlatIndex::stats_info() const {
    VecSimIndexStatsInfo s{};
    s.memory = capacity_ * pitch_ + d_labels_cap_ * 8 + stage_cap_rows_ * pitch_ + id_to_label_.capacity() * sizeof(size_t) +
               (label_to_id_.size() + label_to_ids_.size()) * (sizeof(size_t) + sizeof(void *) * 2 + sizeof(idType));
    return s;
}

static const char *type_name(VecSimType t) {
    switch (t) {
    case VecSimType_FLOAT32: return "FLOAT32";
    case VecSimType_FLOAT64: return "FLOAT64";
    case VecSimType_BFLOAT16: return "BFLOAT16";
    case VecSimType_FLOAT16: return "FLOAT16";
    case VecSimType_INT8: return "INT8";
    case VecSimType_UINT8: return "UINT8";
    case VecSimType_INT32: return "INT32";
    default: return "INT64";
    }
}
static const char *mode_name(VecSearchMode m) { // vec_utils.cpp VecSimSearchMode_ToString
    switch (m) {
    case EMPTY_MODE: return "EMPTY_MODE";
    case STANDARD_KNN: return "STANDARD_KNN";
    case HYBRID_ADHOC_BF: return "HYBRID_ADHOC_BF";
    case HYBRID_BATCHES: return "HYBRID_BATCHES";
    case HYBRID_BATCHES_TO_ADHOC_BF: return "HYBRID_BATCHES_TO_ADHOC_BF";
    default: return "RANGE_QUERY";
    }
}

VecSimIndexDebugInfo FlatIndex::debug_info() const {
    VecSimIndexDebugInfo info;
    memset(&info, 0, sizeof(info));
    info.commonInfo.basicInfo = basic_info();
    info.commonInfo.indexSize = count_;
    info.commonInfo.indexLabelCount = multi_ ? label_to_ids_.size() : label_to_id_.size();
    info.commonInfo.memory = stats_info().memory;
    info.commonInfo.lastMode = last_mode_;
    info.bfInfo.dummy = 0;
    return info;
}

VecSimDebugInfoIterator *FlatIndex::debug_iterator() const {
    auto *it = new VecSimDebugInfoIterator();
    auto str = [&](const char *name, const char *v) {
        VecSim_InfoField f{};
        f.fieldName = name;
        f.fieldType = INFOFIELD_STRING;
        f.fieldValue.stringValue = v;
        it->fields.push_back(f);
    };
    auto u64 = [&](const char *name, uint64_t v) {
        VecSim_InfoField f{};
        f.fieldName = name;
        f.fieldType = INFOFIELD_UINT64;
        f.fieldValue.uintegerValue = v;
        it->fields.push_back(f);
    };
    // order and names: brute_force.h:327-365 + vec_sim_index.h addCommonInfoToIterator
    str("ALGORITHM", "FLAT");
    str("TYPE", type_name(type_));
    u64("DIMENSION", dim_);
    str("METRIC", metric_ == VecSimMetric_L2 ? "L2" : metric_ == VecSimMetric_IP ? "IP" : "COSINE");
    u64("IS_MULTI_VALUE", multi_);
    u64("IS_DISK", 0);
    u64("INDEX_SIZE", count_);
    u64("INDEX_LABEL_COUNT", multi_ ? label_to_ids_.size() : label_to_id_.size());
    u64("MEMORY", stats_info().memory);
    str("LAST_SEARCH_MODE", mode_name(last_mode_));
    u64("BLOCK_SIZE", block_size_);
    return it;
}

int FlatIndex::last_coarse_flags(uint32_t *out, size_t n) {
    std::lock_guard<std::mutex> dg(dev_mu_);
    if (!dev_ctx_ || !last_batch_coarse_ || !dev_ctx_->d_last_ok || dev_ctx_->last_ok_n < n) return -1;
    if (cudaDeviceSynchronize() != cudaSuccess) return -1;
    return cudaMemcpy(out, dev_ctx_->d_last_ok, n * 4, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -1;
}

void set_coarse_mode(int mode) { g_coarse_mode.store(mode); }

// dev_mu_ held.  Folds the CUDA-event timing of the last topk_batch_device scan into the stats.
void FlatIndex::collect_dev_timing_locked() {
    if (!dev_timing_pending_ || !dev_ctx_) return;
    float ms = 0;
    if (cudaEventSynchronize(dev_ctx_->ev_stop) == cudaSuccess &&
        cudaEventElapsedTime(&ms, dev_ctx_->ev_start, dev_ctx_->ev_stop) == cudaSuccess) {
        std::lock_guard<std::mutex> g(stats_mu_);
        scan_us_ += ms * 1000.0;
        scan_launches_++;
        scan_bytes_ += dev_timing_bytes_;
    }
    dev_timing_pending_ = false;
}

VecSimB200_Stats FlatIndex::get_stats(bool reset) {
    {
        std::lock_guard<std::mutex> dg(dev_mu_);
        collect_dev_timing_locked();
    }
    std::lock_guard<std::mutex> g(stats_mu_);
    VecSimB200_Stats s{};
    s.kernel_launches = launches_total_.load();
    s.scan_launches = scan_launches_;
    s.scan_device_us = scan_us_;
    s.scan_bytes = scan_bytes_;
    if (reset) {
        launches_total_ = 0;
        scan_launches_ = 0;
        scan_us_ = 0;
        scan_bytes_ = 0;
    }
    return s;
}

} // namespace rsb200
