// Context, workspace and host<->device staging shared by all translation units of librpk.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/rpk.h"

namespace rpk {

typedef unsigned long long u64;

struct Error : std::runtime_error {
  explicit Error(const std::string& m) : std::runtime_error(m) {}
};

#define RPK_CUDA(call)                                                                             \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      throw rpk::Error(std::string(#call) + " failed: " + cudaGetErrorString(e_) + " (" + __FILE__ + \
                       ":" + std::to_string(__LINE__) + ")");                                      \
  } while (0)

#define RPK_REQUIRE(cond, msg)               \
  do {                                       \
    if (!(cond)) throw rpk::Error(msg);      \
  } while (0)

struct Buf {
  void* p = nullptr;
  size_t cap = 0;
};

enum {
  DBG_WIDE_ACC = 1,    // predict: 64-bit CAS accumulators for every user
  DBG_TINY_LIST = 2,   // selection: smallest legal candidate list
  DBG_MULTI_PASS = 4,  // fit / predict: at least two item-range passes
  DBG_SPLIT_ROWS = 8,  // fit: cut the heaviest rows into pieces even when they are small
  DBG_EXACT_SCORES = 16,  // predict: exact sums for every list even when only the lists are asked for
  DBG_MANY_PASS = 32,     // predict: at least four item ranges
};

}  // namespace rpk

struct rpk_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int64_t launches = 0;
  int flags = 0;
  int dense_users = 0;  // users routed through the tensor-core Gram (-1 = automatic)
  int sm_count = 0;
  int smem_max = 0;  // max opt-in dynamic shared memory per block
  int smem_per_sm = 0;  // shared memory of one SM (CTAs sharing an SM split this, 1 KB reserved each)
  std::map<std::string, rpk::Buf> bufs;
  bool host_out_pending = false;
  // CUDA events around the dominant kernels of the last fit / predict (rpk_last_timings)
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool ev_valid[3] = {false, false, false};
  // side stream for the few heavy rows of a fit (runs next to the main row kernel)
  cudaStream_t side = nullptr;
  cudaEvent_t side_ev[2] = {nullptr, nullptr};
  int last_dense_users = 0;  // users routed to the tensor-core Gram by the last fit
  int last_dense_kd = 0;     // ... padded to the MMA k-block
  void ev_record(int k) {
    if (!ev[k]) RPK_CUDA(cudaEventCreate(&ev[k]));
    RPK_CUDA(cudaEventRecord(ev[k], stream));
  }
  // A fit runs its row range in strips: the tensor-core Gram (k = 0) and the row kernels (k = 1) are timed as the
  // sum of one (begin, end) event pair per strip.
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> spans[2];
  std::vector<cudaEvent_t> span_pool;
  cudaEvent_t span_event() {
    cudaEvent_t e = nullptr;
    if (!span_pool.empty()) {
      e = span_pool.back();
      span_pool.pop_back();
    } else {
      RPK_CUDA(cudaEventCreate(&e));
    }
    RPK_CUDA(cudaEventRecord(e, stream));
    return e;
  }
  void span_reset() {
    for (auto& v : spans) {
      for (auto& pr : v) {
        span_pool.push_back(pr.first);
        if (pr.second) span_pool.push_back(pr.second);
      }
      v.clear();
    }
  }
  void span_begin(int k) { spans[k].emplace_back(span_event(), nullptr); }
  void span_end(int k) { spans[k].back().second = span_event(); }
  // pinned host scratch for small device -> host reads that the host waits for on an event, not on the stream
  int* pinned = nullptr;
  size_t pinned_cap = 0;
  cudaEvent_t hist_ev = nullptr;
  int* pinned_ints(size_t count) {
    if (pinned_cap < count) {
      if (pinned) RPK_CUDA(cudaFreeHost(pinned));
      pinned = nullptr;
      pinned_cap = 0;
      RPK_CUDA(cudaMallocHost(&pinned, sizeof(int) * (count + count / 8 + 64)));
      pinned_cap = count + count / 8 + 64;
    }
    return pinned;
  }
  // strip state of the running fit (see run_fit): the dense / sparse split chosen by strip 0
  int strip_hmax = 0;
  int strip_tau = 32;
  int64_t strip_rows = 0;  // rows per strip, 0 = automatic (rpk_fit_strip_rows)
  // ---- tracing (rpk_trace): named marks on the context's stream, reported as the device time between neighbours
  bool tracing = false;
  std::vector<std::pair<std::string, cudaEvent_t>> marks;
  std::vector<cudaEvent_t> mark_pool;
  std::string trace_text;
  void mark(const char* name) {
    if (!tracing) return;
    cudaEvent_t e = nullptr;
    if (!mark_pool.empty()) {
      e = mark_pool.back();
      mark_pool.pop_back();
    } else {
      RPK_CUDA(cudaEventCreate(&e));
    }
    RPK_CUDA(cudaEventRecord(e, stream));
    marks.emplace_back(name, e);
  }

  // ---- state of the last fit (device pointers into bufs)
  int64_t fit_I = 0;
  // device copies of the last complete fit's lists (valid until the next fit on this context)
  const int32_t* lf_idx = nullptr;
  const double* lf_val = nullptr;
  const int32_t* lf_len = nullptr;
  int64_t lf_I = 0;
  int lf_K = 0;
  int64_t lf_token = 0;  // incremented by every fit

  // ---- loaded model
  int64_t m_I = 0;
  int64_t m_nnz = 0;
  int m_P = 0;        // item-range passes of predict
  int m_R = 0;        // items per pass
  int m_P2 = 0;       // the same for the 32-bit scoring kernel's segment table
  int m_R2 = 0;
  bool m_pad = false;  // padded block layout of the model is current
  int m_max_len = 0;  // longest model row
  int m_exp = 39;     // scale of the loaded model: q = rint(v * 2^m_exp)
  bool m_signed = false;  // the model came from rpk_model_load_signed_csr (float64 scoring, k_predict_signed)
  int64_t filter_I = -1;  // item filter of the predict calls (buffer p_item_ok), -1 = none
  bool pack_flag_pending = false;  // a stream-ordered rpk_model_pack_rows_v left its validation flag unchecked

  // ---- user count of the last rpk_predict_csr_count (rpk_predict_csr_fill must follow it on the same input)
  int64_t pc_U = 0;

  template <class T>
  T* buf(const std::string& name, size_t count) {
    rpk::Buf& b = bufs[name];
    size_t bytes = count * sizeof(T);
    if (bytes == 0) bytes = 16;
    if (b.cap < bytes) {
      if (b.p) RPK_CUDA(cudaFree(b.p));
      b.p = nullptr;
      b.cap = 0;
      size_t want = bytes + bytes / 8 + 256;
      RPK_CUDA(cudaMalloc(&b.p, want));
      b.cap = want;
    }
    return reinterpret_cast<T*>(b.p);
  }
  template <class T>
  T* get(const std::string& name) {
    auto it = bufs.find(name);
    RPK_REQUIRE(it != bufs.end() && it->second.p, "internal: workspace '" + name + "' missing");
    return reinterpret_cast<T*>(it->second.p);
  }
};

namespace rpk {

inline bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Input staging: returns a device pointer holding `count` elements of `p`.
template <class T>
const T* stage_in(rpk_ctx* c, const T* p, size_t count, const char* name) {
  if (count == 0) return c->buf<T>(name, 1);
  RPK_REQUIRE(p != nullptr, std::string("null input pointer: ") + name);
  if (is_device_ptr(p)) return p;
  T* d = c->buf<T>(name, count);
  RPK_CUDA(cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  return d;
}

// Output staging: kernels write to .dev; finish() copies back when the caller's pointer is host memory.
template <class T>
struct Out {
  T* user = nullptr;
  T* dev = nullptr;
  size_t count = 0;
  bool host = false;
  void init(rpk_ctx* c, T* p, size_t n, const char* name) {
    user = p;
    count = n;
    if (!p) {
      dev = nullptr;
      return;
    }
    if (is_device_ptr(p)) {
      dev = p;
      host = false;
    } else {
      dev = c->buf<T>(name, n);
      host = true;
    }
  }
  void finish(rpk_ctx* c) {
    if (user && host && count) {
      RPK_CUDA(cudaMemcpyAsync(user, dev, count * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
      c->host_out_pending = true;
    }
  }
};

inline void finish_call(rpk_ctx* c) {
  if (c->host_out_pending) {
    RPK_CUDA(cudaStreamSynchronize(c->stream));
    c->host_out_pending = false;
  }
}

inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

#define RPK_LAUNCH_CHECK(ctx)          \
  do {                                 \
    (ctx)->launches++;                 \
    RPK_CUDA(cudaGetLastError());      \
  } while (0)

}  // namespace rpk
