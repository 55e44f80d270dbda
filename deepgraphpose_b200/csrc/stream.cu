// Streaming estimate_pose (SURVEY.md 8f rank 2): the reference walks a clip frame by frame (src/deepgraphpose/models/eval.py:
// 256, 306-345: `for frame in clip.iter_frames()` -> sess.run per frame).  Here a reader thread pulls frames from the
// caller's source into a small ring of pinned host slots while the calling thread copies filled slots to the device and
// runs the fused forward + soft-argmax on them; host memory stays bounded by the ring (3 slots of `batch` frames) however
// long the video is, and decode, H2D and compute overlap.
#include "../../include/dgp_b200.h"

#include <cuda_runtime.h>

#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>

#include "handle.cuh"

using namespace dgp;

namespace {

constexpr int kSlots = 3;

struct Ring {
  std::mutex mu;
  std::condition_variable cv;
  bool slot_free[kSlots];
  struct Filled { int slot; int n; const uint8_t* src; };
  std::deque<Filled> filled;
  bool reader_done = false;
  int reader_error = 0;
  bool abort = false;
};

struct ReleaseArg {
  Ring* ring;
  int slot;
};

void CUDART_CB release_slot(void* p) {
  ReleaseArg* a = static_cast<ReleaseArg*>(p);
  {
    std::lock_guard<std::mutex> lk(a->ring->mu);
    a->ring->slot_free[a->slot] = true;
  }
  a->ring->cv.notify_all();
}

// Annotated frames on their way to the writer (dgp_estimate_pose_stream_render): the calling thread takes a free slot before
// it enqueues a batch, the D2H stream hands the slot over once the frames are in it (stream order = video order), and the
// writer thread frees it again after the writer returns.
struct WriterRing {
  std::mutex mu;
  std::condition_variable cv;
  bool slot_free[kSlots];
  struct Ready { int slot; int n; };
  std::deque<Ready> ready;
  bool done = false;  // nothing more will be handed over
  int error = 0;      // first negative return of the writer, or DGP_ERR_CUDA when a slot's packets could not be fetched
  cudaError_t cuda = cudaSuccess;  // the failed packet copy or pinned allocation
  bool overflow = false;           // a JPEG frame above dgp_jpeg_capacity
};

struct HandoffArg {
  WriterRing* ring;
  int slot;
  int n;
};

void CUDART_CB handoff_slot(void* p) {
  HandoffArg* a = static_cast<HandoffArg*>(p);
  {
    std::lock_guard<std::mutex> lk(a->ring->mu);
    a->ring->ready.push_back({a->slot, a->n});
  }
  a->ring->cv.notify_all();
}

// The body of dgp_estimate_pose_stream_transform; with a writer, also that of dgp_estimate_pose_stream_render, and with a
// packet writer that of dgp_estimate_pose_stream_render_jpeg.
int stream_impl(dgp_handle* h, dgp_frame_reader reader, void* user, int H0, int W0, const dgp_frame_transform* transform,
                int batch, float gamma, float gauss_len, int64_t max_frames, float* mu_host, int32_t* peak_host,
                float* lik_host, int64_t* frames_done, const dgp_marker_style* style, dgp_frame_writer writer,
                void* writer_user, int quality = 0, dgp_packet_writer packet_writer = nullptr) {
  if (!h) return DGP_ERR_INVALID;
  if (frames_done) *frames_done = 0;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_estimate_pose_stream before dgp_finalize_weights");
  if (!reader || batch < 1 || max_frames < 0 || !mu_host) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream: bad argument");
  int H, W;
  bool identity;
  if (transform_dims(H0, W0, transform, &H, &W, &identity))
    return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream: invalid frame size or transform");
  const bool jpeg = packet_writer != nullptr;
  const bool render = writer != nullptr || jpeg;
  if (jpeg && (quality < 1 || quality > 100 || jpeg_capacity(H0, W0) < 0))
    return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream_render_jpeg: quality %d or a %dx%d frame outside the JPEG range",
                quality, H0, W0);
  MarkerArgs marker;
  if (render) {
    int rc = marker_args(h, style, H0, W0, &marker);
    if (rc) return rc;
  }
  if (max_frames == 0) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  int rc = h->pose.reserve(h, batch, H0, W0, H, W, identity);
  if (rc) return rc;
  const size_t frame_bytes = (size_t)H0 * W0 * 3;
  for (PinnedBuf& r : h->ring_slot)
    if (r.bytes() < frame_bytes * batch) CU_OK(h, r.alloc(frame_bytes * batch));
  // a writer slot holds a batch's frames, or with JPEG the offsets | sizes of its packets
  const size_t slot_bytes = jpeg ? 2 * sizeof(int64_t) * batch : frame_bytes * batch;
  const int64_t packets_bytes = jpeg ? jpeg_capacity(H0, W0) * batch : 0;
  if (render) {
    if ((rc = h->pose.reserve_render(h, jpeg, batch, marker.trailpoints))) return rc;
    for (PinnedBuf& r : h->writer_slot)
      if (r.bytes() < slot_bytes) CU_OK(h, r.alloc(slot_bytes));
  }
  if (jpeg)
    for (int i = 0; i < kSlots; ++i) {
      if ((rc = ensure(h, &h->jpeg_packets[i], (size_t)packets_bytes))) return rc;
      if ((rc = ensure(h, &h->jpeg_meta[i], 2 * sizeof(int64_t) * batch))) return rc;
    }
  const PoseJob job = {H0, W0, H, W, identity, transform, gamma, gauss_len, mu_host, peak_host, lik_host};

  Ring ring;
  for (int i = 0; i < kSlots; ++i) ring.slot_free[i] = true;
  ReleaseArg rel[kSlots];
  for (int i = 0; i < kSlots; ++i) { rel[i].ring = &ring; rel[i].slot = i; }

  // ---- reader thread: source -> pinned ring
  uint8_t* slots[kSlots];
  for (int i = 0; i < kSlots; ++i) slots[i] = h->ring_slot[i].get<uint8_t>();
  std::thread producer([&ring, &slots, reader, user, batch, max_frames]() {
    int64_t produced = 0;
    while (produced < max_frames) {
      int slot = -1;
      {
        std::unique_lock<std::mutex> lk(ring.mu);
        ring.cv.wait(lk, [&] {
          if (ring.abort) return true;
          for (int i = 0; i < kSlots; ++i) if (ring.slot_free[i]) return true;
          return false;
        });
        if (ring.abort) break;
        for (int i = 0; i < kSlots; ++i) if (ring.slot_free[i]) { slot = i; break; }
        ring.slot_free[slot] = false;
      }
      const int64_t left = max_frames - produced;
      const int want = left < batch ? (int)left : batch;
      const uint8_t* direct = nullptr;
      const int n = reader(user, slots[slot], want, &direct);
      std::lock_guard<std::mutex> lk(ring.mu);
      if (n <= 0 || n > want) {
        ring.slot_free[slot] = true;
        if (n != 0) ring.reader_error = n < 0 ? n : -1;
        break;
      }
      Ring::Filled f;
      f.slot = slot; f.n = n; f.src = direct ? direct : slots[slot];
      ring.filled.push_back(f);
      produced += n;
      ring.cv.notify_all();
    }
    std::lock_guard<std::mutex> lk(ring.mu);
    ring.reader_done = true;
    ring.cv.notify_all();
  });

  // ---- writer thread (rendering only): pinned writer slots -> writer, in video order
  WriterRing wring;
  for (int i = 0; i < kSlots; ++i) wring.slot_free[i] = true;
  HandoffArg hand[kSlots];
  for (int i = 0; i < kSlots; ++i) { hand[i].ring = &wring; hand[i].slot = i; hand[i].n = 0; }
  uint8_t* wslots[kSlots];
  for (int i = 0; i < kSlots; ++i) wslots[i] = h->writer_slot[i].get<uint8_t>();
  std::thread writer_thread;
  // JPEG: the packets of a slot are copied once their total is known (offsets | sizes have arrived in the writer slot)
  auto fetch_packets = [h](WriterRing& wr, int slot, int n, const int64_t* meta) -> const uint8_t* {
    for (int k = 0; k < n; ++k)
      if (meta[n + k] < 0) {
        wr.overflow = true;
        return nullptr;
      }
    const size_t total = (size_t)(meta[n - 1] + meta[2 * n - 1]);
    PinnedBuf& host = h->jpeg_host[slot];
    cudaError_t e = cudaSuccess;
    if (host.bytes() < total) e = host.alloc(total + total / 4);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(host.get(), h->jpeg_packets[slot].get(), total, cudaMemcpyDeviceToHost, h->pose.packet_stream.get());
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->pose.packet_stream.get());
    if (e != cudaSuccess) {
      wr.cuda = e;
      return nullptr;
    }
    return host.get<uint8_t>();
  };
  if (render) {
    writer_thread = std::thread([&wring, &wslots, writer, writer_user, packet_writer, &fetch_packets, h]() {
      if (packet_writer) cudaSetDevice(h->device);  // the pinned packet buffers belong to the handle's device
      for (;;) {
        WriterRing::Ready r;
        {
          std::unique_lock<std::mutex> lk(wring.mu);
          wring.cv.wait(lk, [&] { return !wring.ready.empty() || wring.done; });
          if (wring.ready.empty()) break;
          r = wring.ready.front();
          wring.ready.pop_front();
          if (wring.error) {  // after a failure the remaining slots are released unwritten
            wring.slot_free[r.slot] = true;
            wring.cv.notify_all();
            continue;
          }
        }
        int rc;
        if (packet_writer) {
          const int64_t* meta = reinterpret_cast<const int64_t*>(wslots[r.slot]);
          const uint8_t* data = fetch_packets(wring, r.slot, r.n, meta);
          rc = data ? packet_writer(writer_user, data, meta + r.n, r.n) : DGP_ERR_CUDA;
        } else {
          rc = writer(writer_user, wslots[r.slot], r.n);
        }
        {
          std::lock_guard<std::mutex> lk(wring.mu);
          if (rc < 0 && !wring.error) wring.error = rc;
          wring.slot_free[r.slot] = true;
        }
        wring.cv.notify_all();
      }
    });
  }

  // ---- consumer: H2D (copy stream) -> forward + soft-argmax (compute stream) -> D2H of the read-outs
  int64_t t0 = 0;
  int it = 0;
  bool full_batch_seen = false;
  int status = DGP_OK;
  for (;;) {
    Ring::Filled f;
    {
      std::unique_lock<std::mutex> lk(ring.mu);
      ring.cv.wait(lk, [&] { return !ring.filled.empty() || ring.reader_done; });
      if (ring.filled.empty()) break;
      f = ring.filled.front();
      ring.filled.pop_front();
    }
    // A short batch (the tail of the video, or the wrap of a cyclic source) reuses the full-batch plan once one exists:
    // every frame's arithmetic is independent of its batch, the surplus rows of the device slot hold an earlier batch's
    // frames, and only the first f.n read-outs are copied back.  Building a second plan for it would cost far more than the
    // surplus frames (allocation of every activation, tensor maps, first-use kernel loads).
    const int run_n = (f.n < batch && full_batch_seen) ? batch : f.n;
    if (f.n == batch) full_batch_seen = true;
    RenderBatch rb;
    if (render) {
      int ws = -1;
      {
        std::unique_lock<std::mutex> lk(wring.mu);
        wring.cv.wait(lk, [&] {
          if (wring.error) return true;
          for (int i = 0; i < kSlots; ++i) if (wring.slot_free[i]) return true;
          return false;
        });
        if (wring.error) break;
        for (int i = 0; i < kSlots; ++i) if (wring.slot_free[i]) { ws = i; break; }
        wring.slot_free[ws] = false;
      }
      hand[ws].n = f.n;
      rb = {&marker, wslots[ws], handoff_slot, &hand[ws], jpeg ? quality : 0, h->jpeg_packets[ws].get<uint8_t>(),
            packets_bytes, h->jpeg_meta[ws].get<int64_t>()};
    }
    // the host slot is reusable once its frames have been copied
    if ((status = h->pose.run_batch(h, job, f.src, f.n, run_n, it, t0, release_slot, &rel[f.slot], render ? &rb : nullptr)))
      break;
    t0 += f.n;
    ++it;
  }
  {
    std::lock_guard<std::mutex> lk(ring.mu);
    ring.abort = true;
  }
  ring.cv.notify_all();
  // pending release / hand-off callbacks reference `ring` and `wring`: drain the streams before they go out of scope
  cudaError_t e1 = cudaStreamSynchronize(h->pose.copy_stream.get());
  cudaError_t e2 = cudaStreamSynchronize(h->stream.get());
  const cudaError_t e3 = render ? cudaStreamSynchronize(h->pose.d2h_stream.get()) : cudaSuccess;
  if (e2 == cudaSuccess) e2 = e3;
  producer.join();
  if (render) {
    {
      std::lock_guard<std::mutex> lk(wring.mu);
      wring.done = true;
    }
    wring.cv.notify_all();
    writer_thread.join();
  }
  if (frames_done) *frames_done = t0;
  if (status) return status;
  if (e1 != cudaSuccess || e2 != cudaSuccess)
    return fail(h, DGP_ERR_CUDA, "dgp_estimate_pose_stream: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
  if (ring.reader_error) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream: the frame reader failed (%d)", ring.reader_error);
  if (wring.overflow) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream_render_jpeg: a frame exceeded dgp_jpeg_capacity");
  if (wring.cuda != cudaSuccess)
    return fail(h, DGP_ERR_CUDA, "dgp_estimate_pose_stream_render_jpeg: packet copy: %s", cudaGetErrorString(wring.cuda));
  if (wring.error) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream_render: the frame writer failed (%d)", wring.error);
  return DGP_OK;
}

}  // namespace

extern "C" {

int dgp_cyclic_reader(void* user, uint8_t* slot, int max_frames, const uint8_t** direct) {
  (void)slot;
  dgp_cyclic_source* s = static_cast<dgp_cyclic_source*>(user);
  if (!s || !s->pool || s->pool_frames < 1 || s->frame_bytes == 0) return -1;
  const int64_t left = s->total_frames - s->position;
  if (left <= 0) return 0;
  const int64_t at = s->position % s->pool_frames;
  int64_t n = s->pool_frames - at;
  if (n > max_frames) n = max_frames;
  if (n > left) n = left;
  *direct = s->pool + (size_t)at * s->frame_bytes;
  s->position += n;
  return (int)n;
}

int dgp_estimate_pose_stream(dgp_handle* h, dgp_frame_reader reader, void* user, int H, int W, int batch, float gamma,
                             float gauss_len, int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                             int64_t* frames_done) {
  return dgp_estimate_pose_stream_transform(h, reader, user, H, W, nullptr, batch, gamma, gauss_len, max_frames, mu_host,
                                            peak_host, lik_host, frames_done);
}

int dgp_estimate_pose_stream_transform(dgp_handle* h, dgp_frame_reader reader, void* user, int H0, int W0,
                                       const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                       int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                                       int64_t* frames_done) {
  return stream_impl(h, reader, user, H0, W0, transform, batch, gamma, gauss_len, max_frames, mu_host, peak_host, lik_host,
                     frames_done, nullptr, nullptr, nullptr);
}

int dgp_estimate_pose_stream_render(dgp_handle* h, dgp_frame_reader reader, void* user, int H0, int W0,
                                    const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                    int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                                    int64_t* frames_done, const dgp_marker_style* style, dgp_frame_writer writer,
                                    void* writer_user) {
  if (!h) return DGP_ERR_INVALID;
  if (!writer) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream_render: no frame writer");
  return stream_impl(h, reader, user, H0, W0, transform, batch, gamma, gauss_len, max_frames, mu_host, peak_host, lik_host,
                     frames_done, style, writer, writer_user);
}

int dgp_estimate_pose_stream_render_jpeg(dgp_handle* h, dgp_frame_reader reader, void* user, int H0, int W0,
                                         const dgp_frame_transform* transform, int batch, float gamma, float gauss_len,
                                         int64_t max_frames, float* mu_host, int32_t* peak_host, float* lik_host,
                                         int64_t* frames_done, const dgp_marker_style* style, int quality,
                                         dgp_packet_writer writer, void* writer_user) {
  if (!h) return DGP_ERR_INVALID;
  if (!writer) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream_render_jpeg: no packet writer");
  return stream_impl(h, reader, user, H0, W0, transform, batch, gamma, gauss_len, max_frames, mu_host, peak_host, lik_host,
                     frames_done, style, nullptr, writer_user, quality, writer);
}

}  // extern "C"
