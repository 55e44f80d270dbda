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
  if (!h) return DGP_ERR_INVALID;
  if (frames_done) *frames_done = 0;
  if (!h->finalized) return fail(h, DGP_ERR_STATE, "dgp_estimate_pose_stream before dgp_finalize_weights");
  if (!reader || batch < 1 || max_frames < 0 || !mu_host) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream: bad argument");
  int H, W;
  bool identity;
  if (transform_dims(H0, W0, transform, &H, &W, &identity))
    return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream: invalid frame size or transform");
  if (max_frames == 0) return DGP_OK;
  CU_OK(h, cudaSetDevice(h->device));
  const int nj = h->cfg.num_joints;
  int hf, wf, ho, wo;
  dgp_output_dims(H, W, &hf, &wf, &ho, &wo);
  // the ring, the H2D copy and st_frames2 carry source-size frames; the transform writes st_xf on the compute stream
  const size_t frame_bytes = (size_t)H0 * W0 * 3;
  int rc;
  if ((rc = ensure(h, &h->st_frames2[0], frame_bytes * batch))) return rc;
  if ((rc = ensure(h, &h->st_frames2[1], frame_bytes * batch))) return rc;
  if (!identity && (rc = ensure(h, &h->st_xf, (size_t)H * W * 3 * batch))) return rc;
  if ((rc = ensure(h, &h->st_logits, (size_t)batch * ho * wo * nj * 4))) return rc;
  if ((rc = ensure(h, &h->st_mu, (size_t)batch * nj * 2 * 4))) return rc;
  if ((rc = ensure(h, &h->st_peak, (size_t)batch * nj * 2 * 4))) return rc;
  if ((rc = ensure(h, &h->st_lik, (size_t)batch * nj * 4))) return rc;
  if (h->ring_bytes < frame_bytes * batch) {
    for (int i = 0; i < kSlots; ++i) {
      if (h->ring_slot[i]) cudaFreeHost(h->ring_slot[i]);
      h->ring_slot[i] = nullptr;
    }
    h->ring_bytes = 0;
    for (int i = 0; i < kSlots; ++i) CU_OK(h, cudaHostAlloc(&h->ring_slot[i], frame_bytes * batch, cudaHostAllocDefault));
    h->ring_bytes = frame_bytes * batch;
  }
  if (!h->copy_stream) {
    CU_OK(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      CU_OK(h, cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming));
      CU_OK(h, cudaEventCreateWithFlags(&h->ev_consumed[i], cudaEventDisableTiming));
    }
  }
  cudaStream_t s = h->stream, cs = h->copy_stream;

  Ring ring;
  for (int i = 0; i < kSlots; ++i) ring.slot_free[i] = true;
  ReleaseArg rel[kSlots];
  for (int i = 0; i < kSlots; ++i) { rel[i].ring = &ring; rel[i].slot = i; }

  // ---- reader thread: source -> pinned ring
  uint8_t* slots[kSlots];
  for (int i = 0; i < kSlots; ++i) slots[i] = static_cast<uint8_t*>(h->ring_slot[i]);
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

  // ---- consumer: H2D (copy stream) -> forward + soft-argmax (compute stream) -> D2H of the read-outs
  int64_t t0 = 0;
  int it = 0;
  bool full_batch_seen = false;
  int status = DGP_OK;
  cudaError_t ce = cudaSuccess;
  for (;;) {
    Ring::Filled f;
    {
      std::unique_lock<std::mutex> lk(ring.mu);
      ring.cv.wait(lk, [&] { return !ring.filled.empty() || ring.reader_done; });
      if (ring.filled.empty()) break;
      f = ring.filled.front();
      ring.filled.pop_front();
    }
    const int dslot = it & 1;
    if (it >= 2) ce = cudaStreamWaitEvent(cs, h->ev_consumed[dslot], 0);
    if (ce == cudaSuccess)
      ce = cudaMemcpyAsync(h->st_frames2[dslot].p, f.src, frame_bytes * f.n, cudaMemcpyHostToDevice, cs);
    if (ce == cudaSuccess) ce = cudaLaunchHostFunc(cs, release_slot, &rel[f.slot]);   // the host slot is reusable after the copy
    if (ce == cudaSuccess) ce = cudaEventRecord(h->ev_copied[dslot], cs);
    if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s, h->ev_copied[dslot], 0);
    if (ce != cudaSuccess) break;
    // A short batch (the tail of the video, or the wrap of a cyclic source) reuses the full-batch plan once one exists:
    // every frame's arithmetic is independent of its batch, the surplus rows of the device slot hold an earlier batch's
    // frames, and only the first f.n read-outs are copied back.  Building a second plan for it would cost far more than the
    // surplus frames (allocation of every activation, tensor maps, first-use kernel loads).
    const int run_n = (f.n < batch && full_batch_seen) ? batch : f.n;
    if (f.n == batch) full_batch_seen = true;
    const uint8_t* frames = (const uint8_t*)h->st_frames2[dslot].p;
    if (!identity) {
      if ((status = resize_crop_impl(h, frames, f.n, H0, W0, transform, (uint8_t*)h->st_xf.p, s))) break;
      frames = (const uint8_t*)h->st_xf.p;
    }
    if ((status = dgp_forward(h, frames, run_n, H, W, (float*)h->st_logits.p, nullptr, s))) break;
    if ((ce = cudaEventRecord(h->ev_consumed[dslot], s)) != cudaSuccess) break;
    if ((status = dgp_softargmax(h, (const float*)h->st_logits.p, nullptr, run_n, ho, wo, nj, gamma, gauss_len, (float*)h->st_mu.p,
                                 (int32_t*)h->st_peak.p, (float*)h->st_lik.p, nullptr, nullptr, s)))
      break;
    ce = cudaMemcpyAsync(mu_host + (size_t)t0 * nj * 2, h->st_mu.p, (size_t)f.n * nj * 2 * 4, cudaMemcpyDeviceToHost, s);
    if (ce == cudaSuccess && peak_host)
      ce = cudaMemcpyAsync(peak_host + (size_t)t0 * nj * 2, h->st_peak.p, (size_t)f.n * nj * 2 * 4, cudaMemcpyDeviceToHost, s);
    if (ce == cudaSuccess && lik_host)
      ce = cudaMemcpyAsync(lik_host + (size_t)t0 * nj, h->st_lik.p, (size_t)f.n * nj * 4, cudaMemcpyDeviceToHost, s);
    if (ce != cudaSuccess) break;
    t0 += f.n;
    ++it;
  }
  {
    std::lock_guard<std::mutex> lk(ring.mu);
    ring.abort = true;
  }
  ring.cv.notify_all();
  // pending release callbacks reference `ring`: drain both streams before it goes out of scope
  cudaError_t e1 = cudaStreamSynchronize(cs);
  cudaError_t e2 = cudaStreamSynchronize(s);
  producer.join();
  if (frames_done) *frames_done = t0;
  if (status) return status;
  if (ce != cudaSuccess) return fail(h, DGP_ERR_CUDA, "dgp_estimate_pose_stream: %s", cudaGetErrorString(ce));
  if (e1 != cudaSuccess || e2 != cudaSuccess)
    return fail(h, DGP_ERR_CUDA, "dgp_estimate_pose_stream: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
  if (ring.reader_error) return fail(h, DGP_ERR_INVALID, "dgp_estimate_pose_stream: the frame reader failed (%d)", ring.reader_error);
  return DGP_OK;
}

}  // extern "C"
