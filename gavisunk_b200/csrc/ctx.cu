// ctx.cu -- context life cycle, stream / profiling control, read-batch registration.
#include "common.cuh"

#include <sched.h>
#include <stdlib.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <thread>

extern "C" void gvs_hostpack_range(const uint8_t* ascii, uint64_t n, uint32_t* words, uint64_t w0, uint64_t w1);  // hostpack.cpp

// Host side of the copy/probe pipeline for ASCII host batches.  One submitter thread walks the segments in
// order; each goes out either as it is or packed to 2 bits per base by the pool below (all workers on one
// segment, so that segments finish in order) through the page-locked staging buffer.  gvs_match picks the
// segments up one by one (gvs_pipe_wait) and launches the matching probe variant behind the segment's event.
struct HostPipe {
  // ---- pack pool ----
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_job, cv_done;
  u64 gen = 0;
  bool quit = false;
  int running = 0;
  const u8* ascii = nullptr;
  u64 n = 0;
  u32* words = nullptr;
  u64 w_end = 0;
  std::atomic<u64> next{0};
  static constexpr u64 CHUNK = 1u << 15;  // words per grab: 512 KiB of bases

  void run() {
    for (;;) {
      u64 a = next.fetch_add(CHUNK);
      if (a >= w_end) break;
      u64 b = a + CHUNK < w_end ? a + CHUNK : w_end;
      gvs_hostpack_range(ascii, n, words, a, b);
    }
  }
  void worker(u64 seen) {
    for (;;) {
      {
        std::unique_lock<std::mutex> l(mu);
        cv_job.wait(l, [&] { return quit || gen != seen; });
        if (quit) return;
        seen = gen;
      }
      run();
      {
        std::lock_guard<std::mutex> l(mu);
        if (--running == 0) cv_done.notify_one();
      }
    }
  }
  void start_workers(int n_threads) {
    while ((int)workers.size() < n_threads - 1) workers.emplace_back(&HostPipe::worker, this, gen);  // no job is in flight
  }
  void pack(const u8* a, u64 n_bases, u32* w, u64 w0, u64 w1) {
    {
      std::lock_guard<std::mutex> l(mu);
      ascii = a; n = n_bases; words = w; w_end = w1;
      next.store(w0);
      running = (int)workers.size();
      gen++;
    }
    cv_job.notify_all();
    run();
    std::unique_lock<std::mutex> l(mu);
    cv_done.wait(l, [&] { return running == 0; });
  }
  void stop_workers() {
    {
      std::lock_guard<std::mutex> l(mu);
      quit = true;
    }
    cv_job.notify_all();
    for (auto& t : workers) t.join();
    workers.clear();
    quit = false;
  }

  // ---- submitter ----
  std::thread submitter;
  bool active = false;
  std::mutex smu;
  std::condition_variable scv;
  u64 submitted = 0;  // segments handed to the copy stream
  int err = 0;
  std::string errmsg;
  // ---- page-locked staging for the packed words of the whole batch (grow-only) ----
  u32* stage = nullptr;
  u64 stage_words = 0;
  cudaEvent_t ev_stage_free = nullptr;  // the copies of the previous batch have left the staging buffer
  bool stage_busy = false;
};

static int default_pack_threads() {
  cpu_set_t set;
  int n = 0;
  if (sched_getaffinity(0, sizeof set, &set) == 0) n = CPU_COUNT(&set);
  if (n <= 0) n = (int)std::thread::hardware_concurrency();
  if (n <= 0) n = 1;
  return n > 16 ? 16 : n;
}

int gvs_pipe_join(gvs_ctx* ctx) {
  HostPipe* hp = ctx->pipe;
  if (!hp || !hp->active) return 0;
  hp->submitter.join();
  hp->active = false;
  if (hp->err) return gvs_fail(ctx, hp->err, "%s", hp->errmsg.c_str());
  return 0;
}

int gvs_pipe_wait(gvs_ctx* ctx, u64 seg) {
  HostPipe* hp = ctx->pipe;
  if (!hp || !hp->active) return 0;  // the copies were queued by gvs_reads_set itself
  std::unique_lock<std::mutex> l(hp->smu);
  hp->scv.wait(l, [&] { return hp->err != 0 || hp->submitted > seg; });
  if (hp->err) return gvs_fail(ctx, hp->err, "%s", hp->errmsg.c_str());
  return 0;
}

extern "C" const char* gvs_version(void) { return "gavisunk_b200 0.1 (sm_100a)"; }

extern "C" gvs_ctx* gvs_create(int device, int k) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return nullptr;  // no CPU fallback
  if (k < 1 || k > 32) return nullptr;
  if (cudaSetDevice(device) != cudaSuccess) return nullptr;
  gvs_ctx* c = new gvs_ctx();
  c->device = device;
  c->k = k;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->n_sm = prop.multiProcessorCount;
  for (int i = 0; i < GVS_ST_COUNT; i++) {
    cudaEventCreate(&c->ev0[i]);
    cudaEventCreate(&c->ev1[i]);
    c->ev_valid[i] = false;
  }
  if (gvs_reserve(c, c->counters, 64 * sizeof(u64)) != 0) {
    delete c;
    return nullptr;
  }
  if (cudaHostAlloc(&c->mailbox, 256, cudaHostAllocDefault) != cudaSuccess) c->mailbox = nullptr;  // (read_dev falls back to pageable copies)
  return c;
}

static void release_rows(Rows& r) {
  gvs_release(r.read); gvs_release(r.pos); gvs_release(r.contig);
  gvs_release(r.start); gvs_release(r.group); gvs_release(r.gidx);
}

extern "C" void gvs_destroy(gvs_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->pipe) {
    if (c->pipe->active) c->pipe->submitter.join();
    c->pipe->stop_workers();
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->pipe->stage) cudaFreeHost(c->pipe->stage);
    if (c->pipe->ev_stage_free) cudaEventDestroy(c->pipe->ev_stage_free);
    delete c->pipe;
    c->pipe = nullptr;
  }
  cudaStreamSynchronize(c->stream);
  DevBuf* all[] = {&c->own_words, &c->loc_pack, &c->loc_kmer, &c->loc_contig, &c->loc_start, &c->loc_group, &c->loc_gidx, &c->grp_contig,
                   &c->grp_start, &c->tab_keys, &c->tab_rows, &c->tab_kv, &c->hit_gidx, &c->hit_nf, &c->ohit_gidx, &c->ohit_nf, &c->filt, &c->filt1, &c->contig_hap, &c->contig_hash,
                   &c->contig_len, &c->own_seq, &c->own_off, &c->chunk_first, &c->chunk_hap, &c->tile_first,
                   &c->tile_cnt, &c->tile_off, &c->tile_dst, &c->hit_read, &c->hit_w, &c->hit_row, &c->ohit_read,
                   &c->ohit_w, &c->ohit_row, &c->counters, &c->scan_tmp, &c->scan_tmp2, &c->flags_a, &c->flags_b,
                   &c->flags_c, &c->seg_start, &c->seg_ndist, &c->seg_cap, &c->seg_best, &c->seg_good, &c->seg_dir,
                   &c->diag_scratch, &c->best_read, &c->best_contig, &c->best_good, &c->best_dir, &c->hist,
                   &c->cnt_hist, &c->bad_flag, &c->bad_list, &c->kseg_start, &c->val_scratch, &c->pair_read,
                   &c->pair_contig, &c->pair_group, &c->pair_gidx, &c->parent, &c->present, &c->comp_min, &c->comp_max, &c->comp_cnt, &c->comp_rank, &c->iv_contig, &c->iv_start, &c->iv_end,
                   &c->gap_contig, &c->gap_start, &c->gap_end, &c->nodata_contig, &c->read_len, &c->gt_keys, &c->gt_val,
                   &c->seg_orient, &c->rank_of, &c->rank_grp, &c->sup_diff, &c->pl_strand, &c->pl_tmp,
                   &c->sup_depth, &c->sup_gx, &c->sup_cstat, &c->ge_seg_start, &c->ge_cgap, &c->ge_seg, &c->ge_cand, &c->ge_res,
                   &c->jn_seg_start, &c->jn_row_seg, &c->jn_seg_cnt, &c->jn_flags, &c->jn_scr, &c->dc_diff, &c->dc_scr, &c->dc_seg,
                   &c->pl.buf, &c->sup.buf, &c->ge.buf, &c->jn.buf, &c->dc.buf, &c->dc_runs.buf, &c->rh_scratch, &c->rh.buf,
                   &c->rh_run.buf};
  for (DevBuf* b : all) gvs_release(*b);
  release_rows(c->rows);
  release_rows(c->kept);
  release_rows(c->jn_stash);
  release_rows(c->stash);
  gvs_release(c->stash_len);
  for (int i = 0; i < GVS_ST_COUNT; i++) {
    cudaEventDestroy(c->ev0[i]);
    cudaEventDestroy(c->ev1[i]);
  }
  for (int i = 0; i < 2; i++) {
    if (c->aux[i]) {
      cudaStreamSynchronize(c->aux[i]);
      cudaStreamDestroy(c->aux[i]);
    }
    if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
  }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  for (cudaEvent_t e : c->seg_ev) cudaEventDestroy(e);
  if (c->ev_reads_free) cudaEventDestroy(c->ev_reads_free);
  if (c->copy_stream) {
    cudaStreamSynchronize(c->copy_stream);
    cudaStreamDestroy(c->copy_stream);
  }
  if (c->mailbox) cudaFreeHost(c->mailbox);
  delete c;
}

extern "C" const char* gvs_last_error(gvs_ctx* c) { return c ? c->err.c_str() : "null context (no CUDA device?)"; }

extern "C" int gvs_set_stream(gvs_ctx* ctx, void* s) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->stream = (cudaStream_t)s;
  return 0;
}

extern "C" int gvs_sync(gvs_ctx* ctx) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gvs_set_profiling(gvs_ctx* ctx, int on) {
  if (!ctx) return GVS_E_ARG;
  ctx->profiling = on != 0;
  for (int i = 0; i < GVS_ST_COUNT; i++) ctx->ev_valid[i] = false;
  return 0;
}

extern "C" int gvs_stage_ms(gvs_ctx* ctx, int stage, float* ms) {
  if (!ctx || stage < 0 || stage >= GVS_ST_COUNT || !ms) return GVS_E_ARG;
  if (!ctx->ev_valid[stage]) return gvs_fail(ctx, GVS_E_STATE, "stage %d was not timed", stage);
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventSynchronize(ctx->ev1[stage]));
  CK(cudaEventElapsedTime(ms, ctx->ev0[stage], ctx->ev1[stage]));
  return 0;
}

extern "C" int gvs_set_copy_pipeline(gvs_ctx* ctx, uint64_t min_bytes, uint32_t segments) {
  if (!ctx) return GVS_E_ARG;
  if (segments > 4096) return gvs_fail(ctx, GVS_E_ARG, "at most 4096 copy segments");
  ctx->seg_min_bytes = min_bytes;
  ctx->seg_count = segments;
  ctx->seg_count_set = true;
  return 0;
}

extern "C" int gvs_set_probe_variant(gvs_ctx* ctx, int variant) {
  if (!ctx) return GVS_E_ARG;
  if (variant < 0 || variant > 2) return gvs_fail(ctx, GVS_E_ARG, "probe variant must be 0, 1 or 2");
  ctx->probe_variant = variant;
  return 0;
}

extern "C" int gvs_set_host_pack(gvs_ctx* ctx, int mode, int threads) {
  if (!ctx) return GVS_E_ARG;
  if (mode < GVS_PACK_OFF || mode > GVS_PACK_ALTERNATE) return gvs_fail(ctx, GVS_E_ARG, "unknown host pack mode %d", mode);
  if (threads < 0 || threads > 256) return gvs_fail(ctx, GVS_E_ARG, "host pack threads must be in [0, 256]");
  CKR(gvs_pipe_join(ctx));
  if (ctx->pipe && threads != ctx->pack_threads) ctx->pipe->stop_workers();
  ctx->pack_mode = mode;
  ctx->pack_threads = threads;
  return 0;
}

extern "C" int gvs_copy_stats(gvs_ctx* ctx, uint64_t* h2d_bytes, uint32_t* segments, uint32_t* segments_packed) {
  if (!ctx) return GVS_E_ARG;
  CKR(gvs_pipe_join(ctx));
  if (h2d_bytes) *h2d_bytes = ctx->h2d_bytes;
  if (segments) *segments = ctx->h2d_segs;
  if (segments_packed) *segments_packed = ctx->h2d_segs_packed;
  return 0;
}

extern "C" int gvs_host_alloc(uint64_t bytes, void** p) {
  if (!p) return GVS_E_ARG;
  *p = nullptr;
  if (cudaHostAlloc(p, bytes ? bytes : 16, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    *p = nullptr;
    return GVS_E_NOMEM;
  }
  return 0;
}
extern "C" void gvs_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

extern "C" uint64_t gvs_launch_count(gvs_ctx* ctx) { return ctx ? ctx->launches : 0; }

// Submitter thread of a pipelined ASCII host batch: segment s = tiles [t0, t1) needs the bases of tiles
// [t0, t1 + 2) (the probe's halo) in the buffer of its own kind, so neighbouring segments of different kinds
// overlap by two tiles.
static void host_pipe_main(gvs_ctx* ctx, const u8* seq, u64 total, int mode, bool src_pinned) {
  HostPipe* hp = ctx->pipe;
  auto fail = [&](int code, const char* what, cudaError_t e) {
    std::lock_guard<std::mutex> l(hp->smu);
    hp->err = code;
    hp->errmsg = std::string(what) + ": " + cudaGetErrorString(e);
    hp->scv.notify_all();
  };
  cudaError_t e = cudaSetDevice(ctx->device);
  if (e != cudaSuccess) return fail(GVS_E_CUDA, "cudaSetDevice (copy pipeline)", e);
  const u64 n_seg = ctx->seg_tile_end.size();
  const u64 n_words = cdiv(total, 16);
  using clk = std::chrono::steady_clock;
  // adaptive choice: bytes queued on the link that have not landed yet, retired through the segment events
  std::vector<u64> link_bytes(n_seg, 0);
  u64 inflight = 0, retired = 0;
  double pack_s_per_seg = 0.0;  // last measured pack time of one segment
  const u64 seg_bytes = cdiv(total, n_seg);
  u64 h2d = 0;
  u32 n_packed = 0;
  for (u64 s = 0, t0 = 0; s < n_seg; s++) {
    const u64 t1 = ctx->seg_tile_end[s];
    u64 b0 = t0 * GVS_TILE_BASES, b1 = (t1 + 2) * GVS_TILE_BASES;
    if (b1 > total || s + 1 == n_seg) b1 = total;
    bool pk;
    if (mode == GVS_PACK_ALL || (mode == GVS_PACK_ADAPTIVE && !src_pinned)) {
      pk = true;  // the link cannot read pageable memory by itself: the driver would stage it on one thread
    } else if (mode == GVS_PACK_ALTERNATE) {
      pk = (s & 1) != 0;
    } else {
      while (retired < s && cudaEventQuery(ctx->seg_ev[retired]) == cudaSuccess) inflight -= link_bytes[retired++];
      // keep the link busy for as long as the pool needs for one segment (link taken at 64 GB/s, +25 %),
      // and never fewer than two segments deep
      double need = pack_s_per_seg * 64e9 * 1.25;
      if (need < 2.0 * (double)seg_bytes) need = 2.0 * (double)seg_bytes;
      pk = (double)inflight >= need;
    }
    u64 moved = 0;
    if (b1 > b0) {
      if (pk) {
        const u64 w0 = b0 / 16, w1 = cdiv(b1, 16) < n_words ? cdiv(b1, 16) : n_words;
        auto c0 = clk::now();
        hp->pack(seq, total, hp->stage, w0, w1);
        pack_s_per_seg = std::chrono::duration<double>(clk::now() - c0).count() * (double)seg_bytes / (double)(b1 - b0);
        moved = (w1 - w0) * 4;
        e = cudaMemcpyAsync(ctx->own_words.as<u32>() + w0, hp->stage + w0, moved, cudaMemcpyHostToDevice, ctx->copy_stream);
      } else {
        moved = b1 - b0;
        e = cudaMemcpyAsync((u8*)ctx->own_seq.p + b0, seq + b0, moved, cudaMemcpyHostToDevice, ctx->copy_stream);
      }
      if (e != cudaSuccess) return fail(GVS_E_CUDA, "cudaMemcpyAsync (copy pipeline)", e);
    }
    e = cudaEventRecord(ctx->seg_ev[s], ctx->copy_stream);
    if (e != cudaSuccess) return fail(GVS_E_CUDA, "cudaEventRecord (copy pipeline)", e);
    link_bytes[s] = moved;
    inflight += moved;
    h2d += moved;
    n_packed += pk ? 1 : 0;
    {
      std::lock_guard<std::mutex> l(hp->smu);
      ctx->seg_packed[s] = pk ? 1 : 0;
      hp->submitted = s + 1;
    }
    hp->scv.notify_all();
    t0 = t1;
  }
  ctx->h2d_bytes = h2d;
  ctx->h2d_segs_packed = n_packed;
  if (cudaEventRecord(hp->ev_stage_free, ctx->copy_stream) == cudaSuccess) hp->stage_busy = true;
}

static int start_host_pipe(gvs_ctx* ctx, const u8* seq, u64 total, int mode) {
  if (!ctx->pipe) ctx->pipe = new HostPipe();
  HostPipe* hp = ctx->pipe;
  const u64 n_words = cdiv(total, 16);
  if (!hp->ev_stage_free) CK(cudaEventCreateWithFlags(&hp->ev_stage_free, cudaEventDisableTiming));
  if (hp->stage_busy) {  // recorded before this batch's copies were made to wait for the compute stream
    CK(cudaEventSynchronize(hp->ev_stage_free));
    hp->stage_busy = false;
  }
  if (hp->stage_words < n_words + 16) {
    if (hp->stage) {
      CK(cudaStreamSynchronize(ctx->copy_stream));
      CK(cudaFreeHost(hp->stage));
      hp->stage = nullptr;
      hp->stage_words = 0;
    }
    const u64 want = n_words + n_words / 8 + 64;
    if (cudaHostAlloc((void**)&hp->stage, want * 4, cudaHostAllocDefault) != cudaSuccess) {
      cudaGetLastError();
      hp->stage = nullptr;
      return gvs_fail(ctx, GVS_E_NOMEM, "page-locked staging buffer for %llu packed words", (unsigned long long)want);
    }
    hp->stage_words = want;
  }
  CKR(gvs_reserve(ctx, ctx->own_words, n_words * 4 + 64));
  cudaPointerAttributes at;
  bool src_pinned = cudaPointerGetAttributes(&at, seq) == cudaSuccess && at.type == cudaMemoryTypeHost;
  cudaGetLastError();
  hp->start_workers(ctx->pack_threads > 0 ? ctx->pack_threads : default_pack_threads());
  ctx->seg_packed.assign(ctx->seg_tile_end.size(), 0);
  hp->submitted = 0;
  hp->err = 0;
  hp->errmsg.clear();
  hp->active = true;
  hp->submitter = std::thread(host_pipe_main, ctx, seq, total, mode, src_pinned);
  return 0;
}

// packed: seq holds 2-bit words (16 bases per big-endian u32, zero-padded to a whole word) instead of ASCII
static int reads_set_impl(gvs_ctx* ctx, const uint8_t* seq, bool packed, const uint64_t* read_off, uint64_t n_reads,
                          const uint64_t* chunk_first, const uint8_t* chunk_hap, uint32_t n_chunks, int on_device) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  if (!read_off || !chunk_first || !chunk_hap || n_chunks == 0) return gvs_fail(ctx, GVS_E_ARG, "null read batch arrays");
  if (n_reads >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^32 reads in one batch");
  (void)gvs_pipe_join(ctx);  // a failure of the previous batch's submitter was gvs_match's to report, not this batch's
  ctx->reads_ready = false;
  ctx->match_ready = ctx->diag_ready = ctx->val_ready = false;
  ctx->have_read_len = false;  // lengths come from this batch's offsets, not from an earlier gvs_reads_meta / gvs_batches_bind
  if (chunk_first[0] != 0 || chunk_first[n_chunks] != n_reads) return gvs_fail(ctx, GVS_E_ARG, "chunk_first must span [0, n_reads]");
  for (u32 c = 0; c < n_chunks; c++) {
    if (chunk_first[c] > chunk_first[c + 1]) return gvs_fail(ctx, GVS_E_ARG, "chunk_first not monotone");
    if (chunk_hap[c] > GVS_HAP_ANY) return gvs_fail(ctx, GVS_E_ARG, "chunk haplotype %u (0, 1 or GVS_HAP_ANY)", chunk_hap[c]);
  }
  ctx->h_chunk_first.assign(chunk_first, chunk_first + n_chunks + 1);
  ctx->h_chunk_hap.assign(chunk_hap, chunk_hap + n_chunks);
  ctx->n_chunks = n_chunks;
  CKR(to_dev(ctx, ctx->chunk_first, chunk_first, (size_t)n_chunks + 1));
  CKR(to_dev(ctx, ctx->chunk_hap, chunk_hap, (size_t)n_chunks));
  u64 total = 0;
  if (on_device) {
    if (ctx->copy_stream) CK(cudaStreamSynchronize(ctx->copy_stream));
    ctx->seg_tile_end.clear();
    ctx->seg_packed.clear();
    CKR(read_dev(ctx, read_off + n_reads, &total));
    ctx->seq = seq;
    ctx->read_off = read_off;
  } else {
    total = read_off[n_reads];
    const u64 nbytes = packed ? 4 * cdiv(total, 16) : total;                  // bytes of the sequence buffer
    const u64 tile_bytes = packed ? GVS_TILE_BASES / 4 : GVS_TILE_BASES;      // ... per probe tile
    // 64 bytes of slack: the probe kernel stages 16-byte vectors and may touch the tail
    CKR(gvs_reserve(ctx, ctx->own_seq, nbytes + 64));
    CKR(gvs_reserve(ctx, ctx->own_off, (n_reads + 1) * sizeof(u64)));
    CK(cudaMemcpyAsync(ctx->own_off.p, read_off, (n_reads + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    ctx->seg_tile_end.clear();
    ctx->seg_packed.clear();
    const u64 n_tiles = cdiv(total, GVS_TILE_BASES);
    // ASCII batches large enough for the pipeline may have their segments packed on the host
    int mode = (packed || ctx->k >= 32) ? GVS_PACK_OFF : ctx->pack_mode;  // k = 32 has its own one-kernel match (match.cu)
    u64 n_seg = (nbytes >= ctx->seg_min_bytes && ctx->seg_count > 1) ? ctx->seg_count : 1;
    if (n_seg > 1 && mode != GVS_PACK_OFF && !ctx->seg_count_set) n_seg = GVS_SEG_COUNT_PACK;
    if (n_seg > n_tiles) n_seg = n_tiles ? n_tiles : 1;
    ctx->h2d_bytes = nbytes;
    ctx->h2d_segs = (u32)n_seg;
    ctx->h2d_segs_packed = 0;
    if (n_seg == 1) {
      if (nbytes) CK(cudaMemcpyAsync(ctx->own_seq.p, seq, nbytes, cudaMemcpyHostToDevice, ctx->stream));
    } else {
      if (!ctx->copy_stream) CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
      if (!ctx->ev_reads_free) CK(cudaEventCreateWithFlags(&ctx->ev_reads_free, cudaEventDisableTiming));
      while (ctx->seg_ev.size() < n_seg) {
        cudaEvent_t e;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->seg_ev.push_back(e);
      }
      // the previous batch may still be read by work queued on the compute stream
      CK(cudaEventRecord(ctx->ev_reads_free, ctx->stream));
      CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_reads_free, 0));
      for (u64 s = 0; s < n_seg; s++) ctx->seg_tile_end.push_back((s + 1 == n_seg) ? n_tiles : (s + 1) * n_tiles / n_seg);
      if (mode == GVS_PACK_OFF) {
        u64 c0 = 0;
        for (u64 s = 0; s < n_seg; s++) {
          // the probe prefetches two tiles past the end of its span (the halo of the last windows)
          u64 c1 = (s + 1 == n_seg) ? nbytes : (ctx->seg_tile_end[s] + 2) * tile_bytes;
          if (c1 > nbytes) c1 = nbytes;
          if (c1 > c0) CK(cudaMemcpyAsync((u8*)ctx->own_seq.p + c0, seq + c0, c1 - c0, cudaMemcpyHostToDevice, ctx->copy_stream));
          CK(cudaEventRecord(ctx->seg_ev[s], ctx->copy_stream));
          c0 = c1;
        }
      } else {
        CKR(start_host_pipe(ctx, seq, total, mode));
      }
    }
    ctx->seq = ctx->own_seq.as<u8>();
    ctx->read_off = ctx->own_off.as<u64>();
  }
  ctx->seq_packed = packed;
  ctx->n_reads = n_reads;
  ctx->total_bases = total;
  ctx->reads_ready = true;
  return 0;
}

extern "C" int gvs_reads_set(gvs_ctx* ctx, const uint8_t* seq, const uint64_t* read_off, uint64_t n_reads,
                             const uint64_t* chunk_first, const uint8_t* chunk_hap, uint32_t n_chunks, int on_device) {
  return reads_set_impl(ctx, seq, false, read_off, n_reads, chunk_first, chunk_hap, n_chunks, on_device);
}
extern "C" int gvs_reads_set_packed(gvs_ctx* ctx, const uint32_t* words, const uint64_t* read_off, uint64_t n_reads,
                                    const uint64_t* chunk_first, const uint8_t* chunk_hap, uint32_t n_chunks, int on_device) {
  return reads_set_impl(ctx, (const uint8_t*)words, true, read_off, n_reads, chunk_first, chunk_hap, n_chunks, on_device);
}
