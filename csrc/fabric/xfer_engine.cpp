#include "fabric/xfer_engine.h"

#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>

#include "common/log.h"
#include "common/result.h"
#include "common/tchash_def.h"

namespace bb::gpu {

#define BB_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      BB_LOG(ERROR) << "CUDA error " << cudaGetErrorString(_e) << " (" << static_cast<int>(_e) << ") at " #expr; \
      last_cuda_error_ = static_cast<int>(_e);                                             \
      return ErrorCode::FABRIC_ERROR;                                                      \
    }                                                                                      \
  } while (0)

struct XferEngine::Slot {
  // host (pinned): [descs | tile_start | segment tables (segmented batches)]
  uint8_t* h_tab = nullptr;
  size_t tab_cap = 0;  // bytes of h_tab and d_tab (grown on demand by segmented batches)
  // device
  uint8_t* d_tab = nullptr;
  uint64_t* d_sum = nullptr;
  uint32_t* d_done = nullptr;
  uint64_t* d_digest = nullptr;
  uint32_t* d_status = nullptr;
  // host (pinned) results: [digest | status]
  uint8_t* h_res = nullptr;
  uint32_t* d_debug = nullptr;
  size_t d_debug_bytes = 0;
  uint64_t* d_trace = nullptr;
  size_t d_trace_bytes = 0;
  bool traced = false;
  bool mailed = false;     // served by the resident mailbox warp: results arrive in the mailbox's result ring
  uint32_t mail_first = 0;  // first sequence number of this batch in the mailbox
  bool flagged = false;    // completion by status flag in pinned memory (small-object latency path), no events recorded
  void* stream = nullptr;  // stream of a flagged batch (fallback sync)
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_done = nullptr;
  uint64_t ticket = 0;  // 0 = free
  uint32_t nitems = 0;
  uint32_t ndesc = 0;
  uint32_t total_tiles = 0;
  bool debug = false;
  bool hashed = true;
  uint64_t empty_digest = 0;
  std::vector<int32_t> item_to_desc;  // -1 for zero-size items
};

Result<std::unique_ptr<XferEngine>> XferEngine::create(int device, uint32_t max_items, int slots) {
  std::unique_ptr<XferEngine> e(new XferEngine());
  e->device_ = device;
  e->max_items_ = max_items;
  int prev = 0;
  if (cudaGetDevice(&prev) != cudaSuccess) return ErrorCode::FABRIC_ERROR;
  if (cudaSetDevice(device) != cudaSuccess) return ErrorCode::FABRIC_ERROR;
  const size_t tab_bytes = static_cast<size_t>(max_items) * sizeof(XferDesc) + (static_cast<size_t>(max_items) + 1) * 4;
  const size_t res_bytes = static_cast<size_t>(max_items) * 12;
  bool ok = true;
  for (int i = 0; i < slots && ok; ++i) {
    auto s = std::make_unique<Slot>();
    ok = ok && cudaMallocHost(reinterpret_cast<void**>(&s->h_tab), tab_bytes) == cudaSuccess;
    ok = ok && cudaMallocHost(reinterpret_cast<void**>(&s->h_res), res_bytes) == cudaSuccess;
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&s->d_tab), tab_bytes) == cudaSuccess;
    s->tab_cap = tab_bytes;
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&s->d_sum), static_cast<size_t>(max_items) * 8) == cudaSuccess;
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&s->d_done), static_cast<size_t>(max_items) * 4) == cudaSuccess;
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&s->d_digest), static_cast<size_t>(max_items) * 8) == cudaSuccess;
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&s->d_status), static_cast<size_t>(max_items) * 4) == cudaSuccess;
    ok = ok && cudaMemset(s->d_sum, 0, static_cast<size_t>(max_items) * 8) == cudaSuccess;
    ok = ok && cudaMemset(s->d_done, 0, static_cast<size_t>(max_items) * 4) == cudaSuccess;
    ok = ok && cudaEventCreate(&s->ev_start) == cudaSuccess;
    ok = ok && cudaEventCreate(&s->ev_stop) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&s->ev_done, cudaEventDisableTiming) == cudaSuccess;
    e->slots_.push_back(std::move(s));
  }
  ok = ok && cudaDeviceSynchronize() == cudaSuccess;
  cudaSetDevice(prev);
  if (!ok) {
    BB_LOG(ERROR) << "XferEngine: device allocation failed: " << cudaGetErrorString(cudaGetLastError());
    return ErrorCode::OUT_OF_MEMORY;
  }
  return e;
}

XferEngine::~XferEngine() {
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(device_);
  for (auto& s : slots_) {
    if (s->ev_done) cudaEventSynchronize(s->ev_done);
    cudaFreeHost(s->h_tab);
    cudaFreeHost(s->h_res);
    cudaFree(s->d_tab);
    cudaFree(s->d_sum);
    cudaFree(s->d_done);
    cudaFree(s->d_digest);
    cudaFree(s->d_status);
    if (s->d_debug) cudaFree(s->d_debug);
    if (s->d_trace) cudaFree(s->d_trace);
    if (s->ev_start) cudaEventDestroy(s->ev_start);
    if (s->ev_stop) cudaEventDestroy(s->ev_stop);
    if (s->ev_done) cudaEventDestroy(s->ev_done);
  }
  cudaSetDevice(prev);
}

struct XferEngine::Mailbox {
  MailSlot* slots = nullptr;      // pinned host
  MailResult* results = nullptr;  // pinned host
  MailCtl* ctl = nullptr;         // pinned host
  cudaStream_t stream = nullptr;  // non-blocking: never synchronises with the legacy default stream
  uint32_t next_seq = 1;          // next sequence number to hand out
  uint32_t epoch = 0;             // incarnation counter (0 = never launched)
  uint32_t outstanding = 0;       // posted requests whose results have not been collected
  uint64_t linger_ns = 200000, max_ns = 50000000;
  ~Mailbox() {
    if (stream) {
      cudaStreamSynchronize(stream);  // the resident warp leaves by itself after linger_ns
      cudaStreamDestroy(stream);
    }
    if (slots) cudaFreeHost(slots);
    if (results) cudaFreeHost(results);
    if (ctl) cudaFreeHost(ctl);
  }
};

bool XferEngine::mailbox_enabled() {
  static const bool on = [] {
    const char* e = std::getenv("BB_XFER_MAILBOX");
    return !(e && e[0] == '0');
  }();
  return on && mailbox_on_;
}

ErrorCode XferEngine::mailbox_launch_locked(uint32_t first_seq) {
  Mailbox& m = *mb_;
  ++m.epoch;
  const int rc = launch_mailbox(m.slots, m.results, m.ctl, first_seq, m.epoch, m.linger_ns, m.max_ns, m.stream);
  if (rc != 0) {
    last_cuda_error_ = rc;
    BB_LOG(ERROR) << "launch_mailbox failed: " << cuda_error_string(rc);
    return ErrorCode::FABRIC_ERROR;
  }
  ++mailbox_launches_;
  ++launches_;
  return ErrorCode::OK;
}

// Hands `nd` small single-destination descriptors to the resident warp.  Slot layout and ordering: the 64-byte slot is
// written field by field, the sequence number last (x86 stores stay in order); the warp reads the whole line in one PCIe
// request and acts only when the sequence number is the one it expects.
ErrorCode XferEngine::mailbox_post(Slot* s, const XferDesc* descs, uint32_t nd, int algo) {
  if (!mb_) {
    auto m = std::make_unique<Mailbox>();
    BB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&m->slots), sizeof(MailSlot) * kMailSlots));
    BB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&m->results), sizeof(MailResult) * kMailSlots));
    BB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&m->ctl), sizeof(MailCtl)));
    std::memset(m->slots, 0, sizeof(MailSlot) * kMailSlots);
    std::memset(m->results, 0, sizeof(MailResult) * kMailSlots);
    std::memset(m->ctl, 0, sizeof(MailCtl));
    BB_CUDA(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    if (const char* e = std::getenv("BB_MAILBOX_LINGER_US")) m->linger_ns = static_cast<uint64_t>(std::max(1, std::atoi(e))) * 1000ull;
    mb_ = std::move(m);
  }
  Mailbox& m = *mb_;
  s->mail_first = m.next_seq;
  for (uint32_t i = 0; i < nd; ++i) {
    const uint32_t seq = m.next_seq++;
    MailSlot& q = m.slots[seq % kMailSlots];
    q.src = reinterpret_cast<uint64_t>(descs[i].src);
    q.dst = reinterpret_cast<uint64_t>(descs[i].dst[0]);
    q.expect = descs[i].expect;
    q.nbytes = static_cast<uint32_t>(descs[i].nbytes);
    q.flags = descs[i].flags;
    q.algo = static_cast<uint32_t>(algo);
    q.reserved = descs[i].reserved;
    std::atomic_thread_fence(std::memory_order_release);
    *reinterpret_cast<volatile uint32_t*>(&q.seq) = seq;
  }
  m.outstanding += nd;
  mailbox_requests_ += nd;
  // is anybody polling?  (exit_epoch == epoch: the last incarnation has announced its exit; epoch 0: never launched)
  if (m.epoch == 0 || *reinterpret_cast<volatile uint32_t*>(&m.ctl->exit_epoch) == m.epoch) {
    const uint32_t first = m.epoch == 0 ? s->mail_first : *reinterpret_cast<volatile uint32_t*>(&m.ctl->next_seq);
    return mailbox_launch_locked(first);
  }
  return ErrorCode::OK;
}

ErrorCode XferEngine::mailbox_wait(Slot* s) {
  Mailbox& m = *mb_;
  const uint32_t nd = s->ndesc;
  auto* dg = reinterpret_cast<uint64_t*>(s->h_res);
  auto* stt = reinterpret_cast<uint32_t*>(s->h_res + static_cast<size_t>(max_items_) * 8);
  const auto t0 = std::chrono::steady_clock::now();
  for (uint32_t i = 0; i < nd; ++i) {
    const uint32_t seq = s->mail_first + i;
    const volatile MailResult* r = &m.results[seq % kMailSlots];
    uint32_t spins = 0;
    while (r->seq != seq) {
      if ((++spins & 0x3Fu) != 0) continue;
      // the warp may have left just before our request landed (it lingers only so long): start the next incarnation
      if (*reinterpret_cast<volatile uint32_t*>(&m.ctl->exit_epoch) == m.epoch && r->seq != seq) {
        BB_CUDA(cudaSetDevice(device_));
        const ErrorCode ec = mailbox_launch_locked(*reinterpret_cast<volatile uint32_t*>(&m.ctl->next_seq));
        if (ec != ErrorCode::OK) return ec;
      }
      if ((spins & 0xFFFFu) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::seconds(2)) {
        BB_LOG(ERROR) << "XferEngine: the mailbox warp did not answer request " << seq;
        m.outstanding -= std::min(m.outstanding, nd - i);
        return ErrorCode::FABRIC_ERROR;
      }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    dg[i] = r->digest;
    stt[i] = r->status;
  }
  m.outstanding -= std::min(m.outstanding, nd);
  return ErrorCode::OK;
}

bool XferEngine::flag_completion_enabled() {
  static const bool on = [] {
    const char* e = std::getenv("BB_XFER_FLAG_COMPLETION");
    return !(e && e[0] == '0');
  }();
  return on && flag_completion_;
}

bool XferEngine::small_path_enabled() {
  static const bool on = [] {
    const char* e = std::getenv("BB_XFER_SMALL");
    return !(e && e[0] == '0');
  }();
  return on && small_path_;
}

Result<uint64_t> XferEngine::submit(const std::vector<XferItem>& items, ChecksumAlgo algo, void* stream,
                                    bool capture_debug) {
  if (items.size() > max_items_) return ErrorCode::RESOURCE_EXHAUSTED;
  // pick a free slot (or recycle the oldest finished one)
  Slot* s = nullptr;
  for (auto& c : slots_)
    if (c->ticket == 0) { s = c.get(); break; }
  if (!s) return ErrorCode::RESOURCE_EXHAUSTED;  // caller must wait() on outstanding tickets

  auto run = [&]() -> ErrorCode {
    BB_CUDA(cudaSetDevice(device_));
    // segmented items: their tables follow the descriptor table and tile_start (sized for every item) in the same
    // staging buffer, so the batch is still one H2D copy
    constexpr uint32_t kSegFlags = XFER_GATHER | XFER_SCATTER;
    const size_t seg_base = (items.size() * sizeof(XferDesc) + (items.size() + 1) * 4 + 15) & ~size_t{15};
    uint64_t seg_entries = 0;
    for (const XferItem& it : items)
      if (it.nbytes && (it.flags & kSegFlags)) seg_entries += static_cast<uint64_t>(it.nsegs) + 1;
    const bool segmented = seg_entries > 0;
    if (seg_entries > kMaxSegTableEntries) return ErrorCode::RESOURCE_EXHAUSTED;
    if (segmented && seg_base + seg_entries * sizeof(XferSeg) > s->tab_cap) {
      const size_t cap = std::max<size_t>(seg_base + seg_entries * sizeof(XferSeg), 2 * s->tab_cap);
      cudaFreeHost(s->h_tab);
      cudaFree(s->d_tab);
      s->h_tab = nullptr, s->d_tab = nullptr, s->tab_cap = 0;
      BB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&s->h_tab), cap));
      BB_CUDA(cudaMalloc(reinterpret_cast<void**>(&s->d_tab), cap));
      s->tab_cap = cap;
    }
    auto* seg_h = reinterpret_cast<XferSeg*>(s->h_tab + seg_base);
    uint64_t seg_used = 0;
    // Packs item `it`'s list as one table (header + pieces); returns the table's device address.
    auto pack_segments = [&](const XferItem& it) -> Result<uint64_t> {
      if (!it.segs || it.nsegs == 0) return ErrorCode::INVALID_ARGUMENT;
      XferSeg* t = seg_h + seg_used;
      uint64_t left = it.nbytes, cnt = 0;
      for (uint32_t k = 0; k < it.nsegs && left; ++k) {
        uint64_t p = it.segs[k].ptr, l = it.segs[k].len;
        if (k == 0) {
          if (it.seg_skip >= l) return ErrorCode::INVALID_ARGUMENT;
          p += it.seg_skip, l -= it.seg_skip;
        }
        l = std::min(l, left);
        left -= l;
        if ((p & 15) || (left && (l & 15))) return ErrorCode::INVALID_ADDRESS;
        t[++cnt] = XferSeg{p, it.nbytes - left};
      }
      if (left) return ErrorCode::INVALID_ARGUMENT;
      t[0] = XferSeg{cnt, 0};
      const uint64_t dev = reinterpret_cast<uint64_t>(s->d_tab + seg_base) + seg_used * sizeof(XferSeg);
      seg_used += cnt + 1;
      return dev;
    };
    auto* descs = reinterpret_cast<XferDesc*>(s->h_tab);
    s->item_to_desc.assign(items.size(), -1);
    uint32_t nd = 0, tiles = 0;
    bool all_small = small_path_enabled() && !segmented;
    for (size_t i = 0; i < items.size(); ++i) {
      const XferItem& it = items[i];
      if (it.nbytes == 0) continue;
      all_small = all_small && it.nbytes <= kSmallBytes && !(it.flags & XFER_RAW_SUM) && it.ndst >= 1;
      if (it.ndst > kMaxDst || (it.ndst == 0 && !(it.flags & XFER_RAW_SUM))) return ErrorCode::INVALID_ARGUMENT;
      const bool gather = it.flags & XFER_GATHER, scatter = it.flags & XFER_SCATTER;
      if (scatter && (it.ndst != 1 || (it.flags & XFER_MULTIMEM))) return ErrorCode::INVALID_ARGUMENT;
      uintptr_t al = gather ? 0 : reinterpret_cast<uintptr_t>(it.src);
      for (uint32_t r = scatter ? 1 : 0; r < it.ndst; ++r) al |= reinterpret_cast<uintptr_t>(it.dst[r]);
      if (al & 15) return ErrorCode::INVALID_ADDRESS;
      if ((it.flags & XFER_MULTIMEM) && (it.nbytes & 15)) return ErrorCode::INVALID_ARGUMENT;
      XferDesc& d = descs[nd];
      d.src = it.src;
      for (uint32_t r = 0; r < kMaxDst; ++r) d.dst[r] = r < it.ndst ? it.dst[r] : nullptr;
      if (gather || scatter) {
        auto t = pack_segments(it);
        if (!t.ok()) return t.error();
        if (gather) d.src = reinterpret_cast<const void*>(t.value());
        else d.dst[0] = reinterpret_cast<void*>(t.value());
      }
      d.nbytes = it.nbytes;
      d.first_tile = tiles;
      d.ndst = it.ndst;
      d.expect = it.expect;
      d.flags = it.flags;
      d.reserved = (it.flags & XFER_RAW_SUM) ? it.tile_base : 0;
      if (algo == ChecksumAlgo::CRC32C) {
        d.expect = (static_cast<uint64_t>(crc_init_term_for(it.nbytes)) << 32) | (it.expect & 0xFFFFFFFFull);
        d.reserved = crc_unpad_for(it.nbytes);
      }
      s->item_to_desc[i] = static_cast<int32_t>(nd);
      const uint64_t nt = (it.nbytes + kTileBytes - 1) / kTileBytes;
      if (tiles + nt > 0xFFFFFFF0ull) return ErrorCode::VALUE_OUT_OF_RANGE;
      tiles += static_cast<uint32_t>(nt);
      ++nd;
    }
    auto* tile_start = reinterpret_cast<uint32_t*>(s->h_tab + static_cast<size_t>(nd) * sizeof(XferDesc));
    for (uint32_t i = 0; i < nd; ++i) tile_start[i] = descs[i].first_tile;
    tile_start[nd] = tiles;
    s->nitems = static_cast<uint32_t>(items.size());
    s->ndesc = nd;
    s->total_tiles = tiles;
    s->debug = capture_debug;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nd) {
      const size_t tab = segmented ? seg_base + seg_used * sizeof(XferSeg)
                                   : static_cast<size_t>(nd) * sizeof(XferDesc) + (static_cast<size_t>(nd) + 1) * 4;
      const bool inline_tab = nd <= kInlineDescs && !segmented;
      if (!inline_tab) BB_CUDA(cudaMemcpyAsync(s->d_tab, s->h_tab, tab, cudaMemcpyHostToDevice, st));
      if (capture_debug) {
        const size_t need = static_cast<size_t>(tiles) * tchash::kRows * tchash::kN * 4;
        if (need > s->d_debug_bytes) {
          if (s->d_debug) cudaFree(s->d_debug);
          BB_CUDA(cudaMalloc(reinterpret_cast<void**>(&s->d_debug), need));
          s->d_debug_bytes = need;
        }
      }
      XferLaunch l;
      l.descs = reinterpret_cast<const XferDesc*>(s->d_tab);
      l.tile_start = reinterpret_cast<const uint32_t*>(s->d_tab + static_cast<size_t>(nd) * sizeof(XferDesc));
      l.ndesc = nd;
      l.total_tiles = tiles;
      l.sum_ws = s->d_sum;
      l.done_ws = s->d_done;
      // Small batches: the finalizer warp writes digests / status straight into the pinned result
      // block (UVA), so the launch is the only operation on the stream.
      const bool direct = nd <= kDirectResults;
      l.digest_out = direct ? reinterpret_cast<uint64_t*>(s->h_res) : s->d_digest;
      l.status_out = direct ? reinterpret_cast<uint32_t*>(s->h_res + static_cast<size_t>(max_items_) * 8) : s->d_status;
      if (inline_tab) {
        l.host_descs = descs;
        l.host_tile_start = tile_start;
      }
      l.debug_d = capture_debug ? s->d_debug : nullptr;
      s->traced = tile_trace_;
      if (tile_trace_) {
        const size_t need = static_cast<size_t>(tiles) * 4 * sizeof(uint64_t);
        if (need > s->d_trace_bytes) {
          if (s->d_trace) cudaFree(s->d_trace);
          BB_CUDA(cudaMalloc(reinterpret_cast<void**>(&s->d_trace), need));
          s->d_trace_bytes = need;
        }
        BB_CUDA(cudaMemsetAsync(s->d_trace, 0, need, st));
        l.trace_d = s->d_trace;
      }
      l.algo = algo == ChecksumAlgo::BBH64 ? ALGO_BBH64 : algo == ChecksumAlgo::CRC32C ? ALGO_CRC32C : algo == ChecksumAlgo::XXH3 ? ALGO_XXH3 : ALGO_NONE;
      l.max_ctas = max_ctas_;
      l.stream = stream;
      l.small_path = all_small;
      l.segmented = segmented;
      // Latency path: a small batch whose results land in pinned memory completes by flag -- the launch is the ONLY
      // stream operation (no timing events, no completion event: each costs about as much GPU time as the kernel).
      // (1) resident mailbox warp: no launch at all.  The request bypasses `stream`, so everything already queued there
      // must have finished (the caller's source data is ready), and only one mailed batch is in flight at a time.
      if (all_small && direct && nd <= kMailSlots / 2 && !capture_debug && !tile_trace_ && mailbox_enabled() &&
          (!mb_ || mb_->outstanding == 0)) {
        bool simple = true;
        for (uint32_t i = 0; i < nd; ++i) simple = simple && descs[i].ndst == 1 && !(descs[i].flags & XFER_MULTIMEM);
        if (simple && cudaStreamQuery(st) == cudaSuccess) {
          const ErrorCode mec = mailbox_post(s, descs, nd, l.algo);
          if (mec != ErrorCode::OK) return mec;
          s->mailed = true;
          return ErrorCode::OK;
        }
        cudaGetLastError();  // cudaErrorNotReady is not sticky, but keep the error state clean
      }
      s->flagged = all_small && direct && !capture_debug && !tile_trace_ && flag_completion_enabled();
      if (s->flagged) {
        auto* stt = reinterpret_cast<volatile uint32_t*>(s->h_res + static_cast<size_t>(max_items_) * 8);
        for (uint32_t i = 0; i < nd; ++i) stt[i] = kSmallPending;
        l.flag_completion = true;
        s->stream = stream;
      } else {
        BB_CUDA(cudaEventRecord(s->ev_start, st));
      }
      const int rc = launch_xfer(l);
      if (rc != 0) {
        last_cuda_error_ = rc;
        BB_LOG(ERROR) << "launch_xfer failed: " << cuda_error_string(rc);
        return ErrorCode::FABRIC_ERROR;
      }
      ++launches_;
      if (all_small && !capture_debug && !tile_trace_) ++small_launches_;
      if (s->flagged) return ErrorCode::OK;
      BB_CUDA(cudaEventRecord(s->ev_stop, st));
      if (algo != ChecksumAlgo::NONE && !direct) {
        BB_CUDA(cudaMemcpyAsync(s->h_res, s->d_digest, static_cast<size_t>(nd) * 8, cudaMemcpyDeviceToHost, st));
        BB_CUDA(cudaMemcpyAsync(s->h_res + static_cast<size_t>(max_items_) * 8, s->d_status, static_cast<size_t>(nd) * 4,
                                cudaMemcpyDeviceToHost, st));
      }
    }
    BB_CUDA(cudaEventRecord(s->ev_done, st));
    return ErrorCode::OK;
  };
  s->flagged = false;
  s->mailed = false;
  ErrorCode ec = run();
  if (ec != ErrorCode::OK) return ec;
  s->ticket = next_ticket_++;
  s->hashed = algo != ChecksumAlgo::NONE;
  s->empty_digest = is_tile_sum(algo) ? tchash::finalize(0, 0) : 0;
  return s->ticket;
}

ErrorCode XferEngine::wait(uint64_t ticket, XferResult* out) {
  Slot* s = nullptr;
  for (auto& c : slots_)
    if (c->ticket == ticket) { s = c.get(); break; }
  if (!s) return ErrorCode::NOT_FOUND;
  const uint32_t nd = s->ndesc;
  if (s->mailed) {
    const ErrorCode mec = mailbox_wait(s);
    if (mec != ErrorCode::OK) {
      s->ticket = 0;
      return mec;
    }
  } else if (s->flagged) {
    // spin on the status words the kernel writes last (pinned memory); fall back to a stream sync if they do not show
    // up within a generous bound, so that a launch failure surfaces as an error instead of a hang
    const auto* stt = reinterpret_cast<const volatile uint32_t*>(s->h_res + static_cast<size_t>(max_items_) * 8);
    const auto t0 = std::chrono::steady_clock::now();
    uint32_t done = 0, spins = 0;
    while (done < nd) {
      if (stt[done] != kSmallPending) {
        ++done;
        continue;
      }
      if ((++spins & 0x3FFu) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(200)) {
        BB_CUDA(cudaSetDevice(device_));
        BB_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(s->stream)));
        if (stt[done] == kSmallPending) {
          BB_LOG(ERROR) << "XferEngine: small-object kernel finished without publishing its results";
          s->ticket = 0;
          return ErrorCode::FABRIC_ERROR;
        }
      }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
  } else {
    BB_CUDA(cudaEventSynchronize(s->ev_done));
  }
  const bool no_hash = !s->hashed;
  if (out) {
    out->digest.assign(s->nitems, no_hash ? 0 : s->empty_digest);
    out->status.assign(s->nitems, 0);
    const auto* dg = reinterpret_cast<const uint64_t*>(s->h_res);
    const auto* stt = reinterpret_cast<const uint32_t*>(s->h_res + static_cast<size_t>(max_items_) * 8);
    if (!no_hash) {
      for (uint32_t i = 0; i < s->nitems; ++i) {
        const int32_t d = s->item_to_desc[i];
        if (d >= 0) {
          out->digest[i] = dg[d];
          out->status[i] = stt[d];
        }
      }
    }
    out->device_ms = 0.f;
    if (nd && !s->flagged && !s->mailed) cudaEventElapsedTime(&out->device_ms, s->ev_start, s->ev_stop);
  }
  if (s->debug && nd) {
    debug_host_.resize(static_cast<size_t>(s->total_tiles) * tchash::kRows * tchash::kN);
    BB_CUDA(cudaMemcpy(debug_host_.data(), s->d_debug, debug_host_.size() * 4, cudaMemcpyDeviceToHost));
  }
  if (s->traced && nd) {
    trace_host_.resize(static_cast<size_t>(s->total_tiles) * 4);
    BB_CUDA(cudaMemcpy(trace_host_.data(), s->d_trace, trace_host_.size() * 8, cudaMemcpyDeviceToHost));
  }
  s->ticket = 0;
  return ErrorCode::OK;
}

struct XferEngine::Fp8State {
  uint8_t* h_tab = nullptr;
  uint8_t* d_tab = nullptr;
  uint64_t* d_sum = nullptr;
  uint64_t* h_sum = nullptr;
  uint32_t cap = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ~Fp8State() {
    if (h_tab) cudaFreeHost(h_tab);
    if (h_sum) cudaFreeHost(h_sum);
    if (d_tab) cudaFree(d_tab);
    if (d_sum) cudaFree(d_sum);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

ErrorCode XferEngine::run_fp8(const std::vector<Fp8Item>& items, bool unpack, void* stream, XferResult* out) {
  const uint32_t n = static_cast<uint32_t>(items.size());
  if (n == 0) return ErrorCode::OK;
  if (n > max_items_) return ErrorCode::RESOURCE_EXHAUSTED;
  BB_CUDA(cudaSetDevice(device_));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!fp8_) fp8_ = std::make_unique<Fp8State>();
  Fp8State& f = *fp8_;
  if (f.cap < n) {
    Fp8State fresh;
    const uint32_t cap = std::max<uint32_t>(n, 256);
    const size_t tab = static_cast<size_t>(cap) * sizeof(XferDesc) + (static_cast<size_t>(cap) + 1) * 4;
    BB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&fresh.h_tab), tab));
    BB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&fresh.h_sum), static_cast<size_t>(cap) * 8));
    BB_CUDA(cudaMalloc(reinterpret_cast<void**>(&fresh.d_tab), tab));
    BB_CUDA(cudaMalloc(reinterpret_cast<void**>(&fresh.d_sum), static_cast<size_t>(cap) * 8));
    BB_CUDA(cudaEventCreate(&fresh.ev0));
    BB_CUDA(cudaEventCreate(&fresh.ev1));
    fresh.cap = cap;
    std::swap(f.h_tab, fresh.h_tab), std::swap(f.h_sum, fresh.h_sum), std::swap(f.d_tab, fresh.d_tab), std::swap(f.d_sum, fresh.d_sum);
    std::swap(f.ev0, fresh.ev0), std::swap(f.ev1, fresh.ev1), std::swap(f.cap, fresh.cap);
  }
  auto* descs = reinterpret_cast<XferDesc*>(f.h_tab);
  auto* tile_start = reinterpret_cast<uint32_t*>(f.h_tab + static_cast<size_t>(n) * sizeof(XferDesc));
  uint32_t tiles = 0;
  std::vector<XferItem> scale_items(n);  // scales region of every object, hashed as a RAW_SUM slice by bb_xfer
  for (uint32_t i = 0; i < n; ++i) {
    const Fp8Item& it = items[i];
    if (!fp8_eligible(it.n_elems)) return ErrorCode::INVALID_ARGUMENT;
    if ((reinterpret_cast<uintptr_t>(it.wide) | reinterpret_cast<uintptr_t>(it.packed)) & 15) return ErrorCode::INVALID_ADDRESS;
    const uint32_t nrep = unpack ? 1u : it.nreplicas;
    if (nrep < 1 || nrep > kMaxDst) return ErrorCode::INVALID_ARGUMENT;
    for (uint32_t r = 1; r < nrep; ++r)
      if (!it.more_packed[r - 1] || (reinterpret_cast<uintptr_t>(it.more_packed[r - 1]) & 15)) return ErrorCode::INVALID_ADDRESS;
    auto* payload = static_cast<uint8_t*>(it.packed);
    XferDesc& d = descs[i];
    d.src = unpack ? static_cast<const void*>(payload) : it.wide;
    d.dst[0] = unpack ? it.wide : static_cast<void*>(payload);  // pack: base of the packed object in every replica
    d.dst[1] = nrep > 1 ? it.more_packed[0] : nullptr;
    d.dst[2] = nrep > 2 ? it.more_packed[1] : nullptr;
    d.nbytes = it.n_elems;
    d.first_tile = tiles;
    d.ndst = nrep;
    d.expect = 0;
    d.flags = 0;
    d.reserved = 0;
    tile_start[i] = tiles;
    const uint64_t nt = (it.n_elems + kTileBytes - 1) / kTileBytes;  // payload tiles, the last one possibly partial
    const uint64_t nt_full = it.n_elems / kTileBytes;                // hashed by the fused kernel
    if (tiles + nt > 0xFFFFFFF0ull) return ErrorCode::VALUE_OUT_OF_RANGE;
    tiles += static_cast<uint32_t>(nt);
    // everything past the last whole payload tile (payload tail + scales) is hashed from the stored bytes as a slice
    XferItem& sc = scale_items[i];
    sc.src = payload + nt_full * kTileBytes;
    sc.ndst = 0;
    sc.nbytes = (it.n_elems - nt_full * kTileBytes) + it.n_elems / 32;
    sc.flags = XFER_RAW_SUM;
    sc.tile_base = static_cast<uint32_t>(nt_full);
  }
  tile_start[n] = tiles;
  const size_t tab = static_cast<size_t>(n) * sizeof(XferDesc) + (static_cast<size_t>(n) + 1) * 4;
  BB_CUDA(cudaMemcpyAsync(f.d_tab, f.h_tab, tab, cudaMemcpyHostToDevice, st));
  BB_CUDA(cudaMemsetAsync(f.d_sum, 0, static_cast<size_t>(n) * 8, st));
  XferLaunch l;
  l.descs = reinterpret_cast<const XferDesc*>(f.d_tab);
  l.tile_start = reinterpret_cast<const uint32_t*>(f.d_tab + static_cast<size_t>(n) * sizeof(XferDesc));
  l.ndesc = n;
  l.total_tiles = tiles;
  l.sum_ws = f.d_sum;
  l.max_ctas = max_ctas_;
  l.stream = stream;
  BB_CUDA(cudaEventRecord(f.ev0, st));
  const int rc = launch_xfer_fp8(l, unpack);
  if (rc != 0) {
    last_cuda_error_ = rc;
    BB_LOG(ERROR) << "launch_xfer_fp8 failed: " << cuda_error_string(rc);
    return ErrorCode::FABRIC_ERROR;
  }
  ++launches_;
  BB_CUDA(cudaEventRecord(f.ev1, st));
  BB_CUDA(cudaMemcpyAsync(f.h_sum, f.d_sum, static_cast<size_t>(n) * 8, cudaMemcpyDeviceToHost, st));
  // scales: for a put they were just written by the kernel above (same stream), for a get they are read twice
  XferResult sres;
  ErrorCode ec = run(scale_items, ChecksumAlgo::BBH64, stream, &sres);  // waits for the stream up to here
  if (ec != ErrorCode::OK) return ec;
  BB_CUDA(cudaStreamSynchronize(st));
  if (out) {
    out->digest.assign(n, 0);
    out->status.assign(n, 0);
    for (uint32_t i = 0; i < n; ++i) {
      const uint64_t total = items[i].n_elems + items[i].n_elems / 32;
      out->digest[i] = tchash::finalize(f.h_sum[i] + sres.digest[i], total);
      if (items[i].verify && out->digest[i] != items[i].expect) out->status[i] = 1;
    }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, f.ev0, f.ev1);
    out->device_ms = ms + sres.device_ms;
  }
  return ErrorCode::OK;
}

ErrorCode XferEngine::run(const std::vector<XferItem>& items, ChecksumAlgo algo, void* stream, XferResult* out) {
  auto t = submit(items, algo, stream);
  if (!t.ok()) return t.error();
  return wait(t.value(), out);
}

// ---------------------------------------------------------------- helpers
static int g_dummy_err = 0;
#undef BB_CUDA
#define BB_CUDA_S(expr)                                                                                      \
  do {                                                                                                       \
    cudaError_t _e = (expr);                                                                                 \
    if (_e != cudaSuccess) {                                                                                 \
      BB_LOG(ERROR) << "CUDA error " << cudaGetErrorString(_e) << " at " #expr;                              \
      g_dummy_err = static_cast<int>(_e);                                                                    \
      return ErrorCode::FABRIC_ERROR;                                                                        \
    }                                                                                                        \
  } while (0)

ErrorCode device_count(int* n) {
  *n = 0;
  cudaError_t e = cudaGetDeviceCount(n);
  if (e != cudaSuccess) {
    *n = 0;
    cudaGetLastError();
  }
  return ErrorCode::OK;
}
ErrorCode device_malloc(int device, uint64_t bytes, void** out) {
  BB_CUDA_S(cudaSetDevice(device));
  cudaError_t e = cudaMalloc(out, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return ErrorCode::OUT_OF_MEMORY;
  }
  return ErrorCode::OK;
}
ErrorCode device_free(int device, void* p) {
  BB_CUDA_S(cudaSetDevice(device));
  BB_CUDA_S(cudaFree(p));
  return ErrorCode::OK;
}
ErrorCode host_alloc_pinned(uint64_t bytes, void** out) {
  cudaError_t e = cudaMallocHost(out, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return ErrorCode::OUT_OF_MEMORY;
  }
  return ErrorCode::OK;
}
ErrorCode host_free_pinned(void* p) {
  BB_CUDA_S(cudaFreeHost(p));
  return ErrorCode::OK;
}
ErrorCode stream_synchronize(void* stream) {
  BB_CUDA_S(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return ErrorCode::OK;
}
ErrorCode device_synchronize(int device) {
  BB_CUDA_S(cudaSetDevice(device));
  BB_CUDA_S(cudaDeviceSynchronize());
  return ErrorCode::OK;
}
int device_memcpy_peer_async(void* dst, int dst_device, const void* src, int src_device, uint64_t nbytes, void* stream) {
  return static_cast<int>(cudaMemcpyPeerAsync(dst, dst_device, src, src_device, nbytes, static_cast<cudaStream_t>(stream)));
}
int device_enable_peer_access(int device, int peer) {
  int prev = 0;
  cudaGetDevice(&prev);
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) {
    e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
      cudaGetLastError();
      e = cudaSuccess;
    }
  }
  cudaSetDevice(prev);
  return static_cast<int>(e);
}

const char* cuda_error_string(int code) { return cudaGetErrorString(static_cast<cudaError_t>(code)); }

}  // namespace bb::gpu
