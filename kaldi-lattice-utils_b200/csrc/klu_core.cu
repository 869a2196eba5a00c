// klu_core.cu -- context, buffers, launch bookkeeping and the C ABI entry points
// that are not tool specific.  See include/klu.h for the contract.
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "klu_common.cuh"

namespace klu {

namespace {
__global__ void k_stage_words(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}
void stage_launch(klu_ctx* c, void* dst, const void* src, size_t bytes) {
  const size_t n = bytes / 4;
  const int grid = (int)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, 64));
  k_stage_words<<<grid, 256, 0, c->stream>>>(static_cast<uint32_t*>(dst), static_cast<const uint32_t*>(src), n);
}

// one CTA: L is small next to the arcs
template <typename C, typename O>
__global__ void __launch_bounds__(1024) k_scan_counts(const C* cnt, int l0, int l1, O* off) {
  __shared__ long long warp_sum[32];
  __shared__ long long carry;
  if (threadIdx.x == 0) carry = l0 > 0 ? off[l0] : 0;
  __syncthreads();
  for (int tile = l0; tile < l1; tile += 1024) {
    const int i = tile + threadIdx.x;
    const long long x = cta_exclusive_scan<long long, 1024>(i < l1 ? (long long)cnt[i] : 0, warp_sum, carry);
    if (i < l1) off[i] = x;
  }
  if (threadIdx.x == 0) off[l1] = carry;
}

template <typename C, typename O>
int scan_counts_t(klu_ctx* c, const C* cnt, int l0, int l1, O* off, const char* label) {
  {
    KLU_LAUNCH(c, label);
    k_scan_counts<<<1, 1024, 0, c->stream>>>(cnt, l0, l1, off);
  }
  return check_launch(label);
}
}  // namespace

int scan_counts(klu_ctx* c, const int32_t* cnt, int l0, int l1, int64_t* off, const char* label) {
  return scan_counts_t(c, cnt, l0, l1, off, label);
}
int scan_counts(klu_ctx* c, const long long* cnt, int l0, int l1, long long* off, const char* label) {
  return scan_counts_t(c, cnt, l0, l1, off, label);
}

int stage_begin(klu_ctx* c, size_t L) {
  KLU_CUDA(cudaStreamSynchronize(c->stream));  // nothing in flight reads the area any more
  c->stage_used = 0;
  c->stage_reads.clear();
  const size_t want = 256 * (L + 64) + (64u << 10);
  if (want > c->stage_cap) {
    if (c->h_stage) cudaFreeHost(c->h_stage);
    c->h_stage = nullptr;
    c->stage_cap = 0;
    KLU_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&c->h_stage), want + want / 4, cudaHostAllocDefault));
    c->stage_cap = want + want / 4;
  }
  return 0;
}

int small_h2d(klu_ctx* c, void* dst_dev, const void* src_host, size_t bytes) {
  if (!bytes) return 0;
  const size_t need = (bytes + 15) & ~(size_t)15;
  if ((bytes & 3) || c->stage_used + need > c->stage_cap) {
    KLU_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, c->stream));
    return 0;
  }
  char* st = c->h_stage + c->stage_used;
  c->stage_used += need;
  memcpy(st, src_host, bytes);
  stage_launch(c, dst_dev, st, bytes);
  KLU_CUDA(cudaGetLastError());
  return 0;
}

int small_d2h(klu_ctx* c, void* dst_host, const void* src_dev, size_t bytes) {
  if (!bytes) return 0;
  const size_t need = (bytes + 15) & ~(size_t)15;
  if ((bytes & 3) || c->stage_used + need > c->stage_cap) {
    KLU_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, c->stream));
    return 0;
  }
  const size_t off = c->stage_used;
  c->stage_used += need;
  stage_launch(c, c->h_stage + off, src_dev, bytes);
  KLU_CUDA(cudaGetLastError());
  c->stage_reads.push_back({dst_host, off, bytes});
  return 0;
}

int small_sync(klu_ctx* c) {
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  for (const auto& r : c->stage_reads) memcpy(r.dst, c->h_stage + r.off, r.bytes);
  c->stage_reads.clear();
  return 0;
}

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }

int DevBuf::reserve(size_t bytes) {
  if (bytes <= cap) return 0;
  if (p) {
    cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  size_t want = bytes + bytes / 8 + 256;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    e = cudaMalloc(&p, bytes);
    want = bytes;
  }
  if (e != cudaSuccess) {
    set_error(std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
    p = nullptr;
    return 1;
  }
  cap = want;
  return 0;
}

void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}

LaunchScope::LaunchScope(klu_ctx* ctx, const char* n) : c(ctx), name(n) {
  c->launches++;
  if (c->profile) {
    auto get = [&]() {
      cudaEvent_t e;
      if (!c->event_pool.empty()) {
        e = c->event_pool.back();
        c->event_pool.pop_back();
      } else {
        cudaEventCreate(&e);
      }
      return e;
    };
    a = get();
    b = get();
    cudaEventRecord(a, c->stream);
  }
}

LaunchScope::~LaunchScope() {
  if (c->profile && a) {
    cudaEventRecord(b, c->stream);
    c->prof_pending.push_back(std::make_pair(std::string(name), std::make_pair(a, b)));
  }
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error(std::string(what) + ": " + cudaGetErrorString(e));
    return 1;
  }
  return 0;
}

CostParams make_cost_params(const klu_opts* o, bool float_sum) {
  CostParams cp;
  cp.gs = (double)o->graph_scale;
  cp.as = (double)o->acoustic_scale;
  cp.gsf = o->graph_scale;
  cp.asf = o->acoustic_scale;
  cp.pen = o->insertion_penalty;
  cp.scale = (o->acoustic_scale != 1.0f || o->graph_scale != 1.0f) ? 1 : 0;
  cp.float_sum = float_sum ? 1 : 0;
  return cp;
}

// Label filter (kwsbin2/lattice-word-index-position.cc:150-155): mode 0 = none,
// 1 = include list, 2 = exclude list; sorted unique labels on the device.
int upload_filter(klu_ctx* c, const klu_opts* o, int* mode_out, int* n_out) {
  std::vector<int32_t> v;
  int mode = 0;
  if (o->num_include > 0) {
    mode = 1;
    v.assign(o->include_words, o->include_words + o->num_include);
  } else if (o->num_exclude > 0) {
    mode = 2;
    v.assign(o->exclude_words, o->exclude_words + o->num_exclude);
  }
  std::sort(v.begin(), v.end());
  v.erase(std::unique(v.begin(), v.end()), v.end());
  if (!v.empty()) {
    KLU_TRY(c->d_filter.reserve(v.size() * sizeof(int32_t)));
    KLU_CUDA(cudaMemcpyAsync(c->d_filter.p, v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    KLU_CUDA(cudaStreamSynchronize(c->stream));  // v goes out of scope
  }
  *mode_out = mode;
  *n_out = (int)v.size();
  return 0;
}

}  // namespace klu

klu::BatchView klu_ctx::view() const {
  klu::BatchView v;
  v.L = L;
  v.S = (int32_t)S;
  v.E = (int32_t)E;
  v.s_off = d_s_off.as<int32_t>();
  v.e_off = d_e_off.as<int32_t>();
  v.lvl_off = d_lvl_off.as<int32_t>();
  v.lvl_start = d_lvl_start.as<int32_t>();
  v.in_rec = d_in_rec.as<int4>();
  v.out_rec = d_out_rec.as<int4>();
  v.in_off = d_in_off.as<int32_t>();
  v.out_off = d_out_off.as<int32_t>();
  v.out_src = d_out_src.as<int32_t>();
  v.out_orig = d_out_orig.as<int32_t>();
  v.in2out = d_in2out.as<int32_t>();
  v.fin_g = d_fin_g.as<float>();
  v.fin_a = d_fin_a.as<float>();
  v.time = d_time.as<int32_t>();
  v.orig = d_orig.as<int32_t>();
  v.old2new = d_old2new.as<int32_t>();
  v.level = d_level.as<int32_t>();
  v.band_lo = d_band_lo.as<int32_t>();
  v.band_off = d_band_off.as<int64_t>();
  v.order = d_order.as<int32_t>();
  v.fr_base = d_fr_base.as<int32_t>();
  v.fr_off = d_fr_off.as<int64_t>();
  v.frame_arc = d_frame_arc.as<int32_t>();
  return v;
}

using namespace klu;

extern "C" {

const char* klu_last_error(void) { return g_error.c_str(); }
int klu_version(void) { return KLU_VERSION; }

void klu_opts_default(klu_opts* o) {
  memset(o, 0, sizeof(*o));
  o->acoustic_scale = 1.0f;
  o->graph_scale = 1.0f;
  o->insertion_penalty = 0.0f;
  o->beam = INFINITY;
  o->beam_ratio = 0.9f;
  o->min_beam = 1e-3f;
  o->max_arcs = INT_MAX;
  o->max_states = INT_MAX;
  o->nbest = 100;
}

int klu_device_count(int* n) {
  *n = 0;
  cudaError_t e = cudaGetDeviceCount(n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error(std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    *n = 0;
    return 1;
  }
  return 0;
}

int klu_create(int device, klu_ctx** out) {
  *out = nullptr;
  int n = 0;
  if (klu_device_count(&n) != 0 || n <= 0) {
    if (g_error.empty()) set_error("no CUDA device: this library has no CPU fallback");
    return 1;
  }
  if (device < 0 || device >= n) {
    set_error("invalid device index");
    return 1;
  }
  KLU_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  KLU_CUDA(cudaGetDeviceProperties(&prop, device));
  klu_ctx* c = new klu_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  auto init = [&]() -> int {
    KLU_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    KLU_CUDA(cudaEventCreate(&c->ev0));
    KLU_CUDA(cudaEventCreate(&c->ev1));
    KLU_CUDA(cudaEventCreate(&c->ev_p0));
    KLU_CUDA(cudaEventCreate(&c->ev_p1));
    return 0;
  };
  if (init() != 0) {  // nothing of a half-made context is left behind
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev_p0) cudaEventDestroy(c->ev_p0);
    if (c->ev_p1) cudaEventDestroy(c->ev_p1);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 1;
  }
  *out = c;
  return 0;
}

int klu_destroy(klu_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  DevBuf* bufs[] = {&c->d_s_off, &c->d_e_off, &c->d_lvl_off, &c->d_lvl_start, &c->d_in_rec, &c->d_out_rec,
                    &c->d_in_off, &c->d_out_off, &c->d_out_src, &c->d_out_orig, &c->d_in2out, &c->d_old2new, &c->d_fin_g, &c->d_fin_a,
                    &c->d_time, &c->d_orig, &c->d_level, &c->d_band_lo, &c->d_band_off, &c->d_order, &c->d_fr_base, &c->d_fr_off, &c->d_frame_arc, &c->d_fr_item, &c->d_fr_gloc, &c->d_fr_res_off, &c->d_fr_gword, &c->d_fr_gstart, &c->d_fr_gframe, &c->d_fr_run_lo, &c->d_fr_run_hi, &c->d_fr_tarc, &c->d_fr_tlabel, &c->d_fr_seg, &c->d_tile_heads, &c->d_sg_meta, &c->d_sg_boff, &c->d_sg_perm, &c->d_sortws, &c->d_alpha, &c->d_beta,
                    &c->d_total, &c->d_totfwd, &c->d_counter, &c->d_filter, &c->d_vfwd, &c->d_vbwd, &c->d_best,
                    &c->d_alpha2, &c->d_flush};
  char_release(c);
  for (DevBuf* b : bufs) b->release();
  for (auto& b : c->d_scratch) b.release();
  for (auto& b : c->d_res) b.release();
  for (auto e : c->event_pool) cudaEventDestroy(e);
  for (auto& p : c->prof_pending) {
    cudaEventDestroy(p.second.first);
    cudaEventDestroy(p.second.second);
  }
  cudaEventDestroy(c->ev0);
  cudaEventDestroy(c->ev1);
  cudaEventDestroy(c->ev_p0);
  cudaEventDestroy(c->ev_p1);
  if (c->h_stage) cudaFreeHost(c->h_stage);
  cudaStreamDestroy(c->stream);
  delete c;
  return 0;
}

int klu_host_alloc(size_t bytes, void** out) {
  *out = nullptr;
  KLU_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  return 0;
}

int klu_host_free(void* p) {
  if (p) KLU_CUDA(cudaFreeHost(p));
  return 0;
}

int klu_load(klu_ctx* c, const klu_lattices* lats) {
  KLU_CUDA(cudaSetDevice(c->device));
  c->loaded = false;
  c->last_tool = -1;
  if (lats->num_lattices < 0) {
    set_error("klu_load: negative lattice count");
    return 1;
  }
  for (int32_t l = 0; l < lats->num_lattices; ++l)  // negative sizes must not reach the kernels
    if (lats->state_off[l + 1] < lats->state_off[l] || lats->arc_off[l + 1] < lats->arc_off[l]) {
      set_error("klu_load: lattice " + std::to_string(l) + ": state_off / arc_off must be non-decreasing");
      return 1;
    }
  c->h_frame_res_off.assign(1, 0);
  c->fr_items = 0;
  klu_lattices with_src;
  std::vector<int32_t> src_tmp, dst_tmp, dur_tmp, label_tmp;
  if (!lats->arc_dst && !lats->arc_dst_delta_u16) {
    set_error("klu_load: arc_dst and arc_dst_delta_u16 are both NULL");
    return 1;
  }
  if (!lats->arc_dur && !lats->arc_dur_u8) {
    set_error("klu_load: arc_dur and arc_dur_u8 are both NULL");
    return 1;
  }
  if (!lats->arc_label && !lats->arc_label_u16) {
    set_error("klu_load: arc_label and arc_label_u16 are both NULL");
    return 1;
  }
  if (!lats->arc_src) {
    if (!lats->state_num_arcs) {
      set_error("klu_load: arc_src and state_num_arcs are both NULL");
      return 1;
    }
    for (int32_t l = 0; l < lats->num_lattices; ++l) {  // the counts must tile each lattice's arc range
      int64_t sum = 0;
      for (int64_t s = lats->state_off[l]; s < lats->state_off[l + 1]; ++s) {
        if (lats->state_num_arcs[s] < 0) sum = -1;
        if (sum < 0) break;
        sum += lats->state_num_arcs[s];
      }
      if (sum != lats->arc_off[l + 1] - lats->arc_off[l]) {
        set_error("klu_load: lattice " + std::to_string(l) + ": state_num_arcs does not add up to its arc count");
        return 1;
      }
    }
    if (getenv("KLU_HOST_PACKER")) {  // the host twin wants explicit sources
      src_tmp.resize((size_t)lats->arc_off[lats->num_lattices]);
      for (int32_t l = 0; l < lats->num_lattices; ++l) {
        int64_t e = lats->arc_off[l];
        for (int64_t s = lats->state_off[l]; s < lats->state_off[l + 1]; ++s)
          for (int32_t k = 0; k < lats->state_num_arcs[s]; ++k) src_tmp[(size_t)e++] = (int32_t)(s - lats->state_off[l]);
      }
      with_src = *lats;
      with_src.arc_src = src_tmp.data();
      lats = &with_src;
    }
  }
  if (getenv("KLU_HOST_PACKER") && (!lats->arc_dst || !lats->arc_dur || !lats->arc_label)) {  // the host twin wants 32-bit arrays
    const size_t E = (size_t)lats->arc_off[lats->num_lattices];
    if (lats != &with_src) {
      with_src = *lats;
      lats = &with_src;
    }
    if (!with_src.arc_dst) {
      dst_tmp.resize(E);
      for (size_t e = 0; e < E; ++e) dst_tmp[e] = with_src.arc_src[e] + (int32_t)with_src.arc_dst_delta_u16[e];
      with_src.arc_dst = dst_tmp.data();
    }
    if (!with_src.arc_dur) {
      dur_tmp.resize(E);
      for (size_t e = 0; e < E; ++e) dur_tmp[e] = (int32_t)with_src.arc_dur_u8[e];
      with_src.arc_dur = dur_tmp.data();
    }
    if (!with_src.arc_label) {
      label_tmp.resize(E);
      for (size_t e = 0; e < E; ++e) label_tmp[e] = (int32_t)with_src.arc_label_u16[e];
      with_src.arc_label = label_tmp.data();
    }
  }
  c->load_upload_ms = c->load_pack_ms = c->lazy_pack_ms = 0.f;
  c->frame_ready = false;
  c->seg_ready = false;
  if (getenv("KLU_HOST_PACKER")) {
    KLU_TRY(pack_and_upload(c, lats));  // builds the frame index as it goes
    c->frame_ready = true;
  } else {
    KLU_TRY(pack_and_upload_gpu(c, lats));
  }
  c->loaded = true;
  klu_trace(c, "load: done");
  return 0;
}

int klu_run(klu_ctx* c, int tool, const klu_opts* opts) {
  if (!c->loaded) {
    set_error("klu_run: no batch loaded");
    return 1;
  }
  KLU_CUDA(cudaSetDevice(c->device));
  klu_opts def;
  if (!opts) {
    klu_opts_default(&def);
    opts = &def;
  }
  c->last_tool = -1;
  c->frame_col_static = false;
  int rc = 0;
  switch (tool) {
    case KLU_FRAME_POST:
      // frame-synchronous kernel; KLU_GENERIC_FRAME_POST=1 selects the generic
      // emit/sort/reduce pipeline instead (kept as a cross-check)
      rc = getenv("KLU_GENERIC_FRAME_POST") ? run_index_tool(c, tool, opts) : run_frame_post(c, opts);
      break;
    case KLU_SEGMENT: {
      // arcs bucketed by start frame; KLU_GENERIC_SEGMENT=1 (or a bucket over the cap) selects the
      // generic emit/sort/reduce pipeline instead (kept as a cross-check)
      bool done = false;
      rc = run_segment_buckets(c, opts, &done);
      if (rc == 0 && !done) rc = run_index_tool(c, tool, opts);
      break;
    }
    case KLU_FWD_BWD:
    case KLU_UTTERANCE:
      rc = run_index_tool(c, tool, opts);
      break;
    case KLU_POSITION:
    case KLU_POSITION_POST:
      // (word, position) cells; KLU_GENERIC_POSITION=1 selects the generic emit/sort/reduce
      // pipeline over one entry per (arc, length) instead (kept as a cross-check)
      rc = getenv("KLU_GENERIC_POSITION") ? run_index_tool(c, tool, opts) : run_position_tool(c, tool, opts);
      break;
    case KLU_BEST_PATH2:
      rc = run_position_tool(c, tool, opts);
      break;
    case KLU_PRUNE_DYN_BEAM:
      rc = run_prune_dyn_beam(c, opts);
      break;
    case KLU_PRUNE_ARCS:
      rc = run_prune_arcs(c, opts);
      break;
    case KLU_CHAR_POSITION:
      rc = run_char_position(c, opts);
      break;
    case KLU_CHAR_SEGMENT:
      rc = run_char_segment(c, opts);
      break;
    case KLU_LENGTH_DIST:
      rc = run_length_dist(c, opts);
      break;
    default:
      set_error("klu_run: unknown tool");
      return 1;
  }
  if (rc == 0) c->last_tool = tool;
  return rc;
}

int klu_sync(klu_ctx* c) {
  KLU_CUDA(cudaSetDevice(c->device));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int klu_timer_start(klu_ctx* c) {
  KLU_CUDA(cudaSetDevice(c->device));
  KLU_CUDA(cudaEventRecord(c->ev0, c->stream));
  return 0;
}

int klu_timer_stop(klu_ctx* c, float* ms) {
  KLU_CUDA(cudaSetDevice(c->device));
  KLU_CUDA(cudaEventRecord(c->ev1, c->stream));
  KLU_CUDA(cudaEventSynchronize(c->ev1));
  KLU_CUDA(cudaEventElapsedTime(ms, c->ev0, c->ev1));
  return 0;
}

int klu_launch_count(klu_ctx* c, int64_t* n) {
  *n = c->launches;
  return 0;
}

int klu_profile_enable(klu_ctx* c, int on) {
  c->profile = on != 0;
  if (on) c->prof.clear();
  return 0;
}

int klu_profile_json(klu_ctx* c, char* buf, size_t cap) {
  KLU_CUDA(cudaSetDevice(c->device));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  for (auto& p : c->prof_pending) {
    float ms = 0;
    cudaEventElapsedTime(&ms, p.second.first, p.second.second);
    auto& st = c->prof[p.first];
    st.launches++;
    st.ms += ms;
    c->event_pool.push_back(p.second.first);
    c->event_pool.push_back(p.second.second);
  }
  c->prof_pending.clear();
  std::string s = "{";
  bool first = true;
  for (auto& kv : c->prof) {
    if (!first) s += ", ";
    first = false;
    char tmp[256];
    snprintf(tmp, sizeof(tmp), "\"%s\": {\"launches\": %lld, \"ms\": %.6f}", kv.first.c_str(),
             (long long)kv.second.launches, kv.second.ms);
    s += tmp;
  }
  s += "}";
  if (s.size() + 1 > cap) {
    set_error("klu_profile_json: buffer too small");
    return 1;
  }
  memcpy(buf, s.c_str(), s.size() + 1);
  return 0;
}

int klu_load_times(klu_ctx* c, float* upload_ms, float* pack_ms, float* frame_index_ms) {
  if (upload_ms) *upload_ms = c->load_upload_ms;
  if (pack_ms) *pack_ms = c->load_pack_ms;
  if (frame_index_ms) *frame_index_ms = c->lazy_pack_ms;
  return 0;
}

int klu_batch_stats(klu_ctx* c, int64_t stats[8]) {
  stats[0] = c->L;
  stats[1] = c->S;
  stats[2] = c->E;
  stats[3] = c->NL;
  stats[4] = c->last_entries;
  stats[5] = c->band_total;
  stats[6] = c->frame_entries;
  stats[7] = c->max_time;
  return 0;
}

__global__ void k_flush(int4* p, size_t n, int v) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = make_int4(v, v, v, v);
}

int klu_flush_l2(klu_ctx* c) {
  KLU_CUDA(cudaSetDevice(c->device));
  const size_t bytes = (size_t)256 << 20;  // 2x the 126 MB L2
  KLU_TRY(c->d_flush.reserve(bytes));
  static int v = 0;
  k_flush<<<c->num_sms * 4, 256, 0, c->stream>>>(c->d_flush.as<int4>(), bytes / sizeof(int4), ++v);
  return check_launch("k_flush");
}

}  // extern "C"
