// b200z_api.cu -- the C ABI (include/b200z.h): context, staging, and the host-side framing logic
// that sits between the reference's codec classes and the kernels.
//
// Host logic restated here (reference, paths relative to /root/reference/):
//   lib/src/codecs/zlib/_gzip_decoder_web.dart:27-138   member loop + header skip
//   lib/src/codecs/zlib/_zlib_decoder_web.dart:31-107   stream loop + FCHECK/FDICT + Adler verify
// The byte-level work (Huffman decode, LZ77, Adler-32) runs on the GPU; nothing here decodes.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "b200z_internal.h"
#include "bzip2_enc.h"

namespace b200z {

static thread_local char t_err[512] = "";
static void set_err(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof t_err, fmt, ap);
  va_end(ap);
}

static std::atomic<uint64_t> g_launches{0};
static std::atomic<unsigned long long> g_bz2_fast_blocks{0}, g_bz2_exact_blocks{0};  // K7: blocks by the fast / the exact kernel
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + (n >> 3) + 4096;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      p = nullptr;
      return e;
    }
    cap = want;
    return cudaSuccess;
  }
  // grow but keep the first `keep` bytes (decoded members already sitting in the buffer)
  cudaError_t reserve_keep(size_t n, size_t keep, cudaStream_t s) {
    if (n <= cap) return cudaSuccess;
    size_t want = n + (n >> 2) + 4096;
    void *np = nullptr;
    cudaError_t e = cudaMalloc(&np, want);
    if (e != cudaSuccess) return e;
    if (p && keep) {
      e = cudaMemcpyAsync(np, p, keep < cap ? keep : cap, cudaMemcpyDeviceToDevice, s);
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
      if (e != cudaSuccess) {
        cudaFree(np);
        return e;
      }
    }
    if (p) cudaFree(p);
    p = np;
    cap = want;
    return cudaSuccess;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};
struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = n + (n >> 2) + 4096;
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
    if (e != cudaSuccess) {
      p = nullptr;
      return e;
    }
    cap = want;
    return cudaSuccess;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

struct Ctx {
  std::mutex mu;
  bool inited = false;
  int device = -1;
  cudaStream_t stream = nullptr, s_h2d = nullptr, s_d2h = nullptr;
  static const int kCompStreams = 8;
  cudaStream_t s_comp[kCompStreams] = {};
  DevBuf d_in, d_out, d_ws, d_meta, d_small, d_bz, d_tok;
  PinBuf h_meta;
};
static Ctx g;

#define CU(x)                                                                       \
  do {                                                                              \
    cudaError_t e__ = (x);                                                          \
    if (e__ != cudaSuccess) {                                                       \
      set_err("%s failed: %s (%s:%d)", #x, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return B200Z_E_NODEVICE;                                                      \
    }                                                                               \
  } while (0)

static int require_init() {
  if (!g.inited) {
    set_err("b200z_init has not been called (or no CUDA device): there is no CPU fallback");
    return B200Z_E_NODEVICE;
  }
  return B200Z_OK;
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------
// Adler-32 on the device (adler32.dart:29-52).  s1 = 1 + sum b_i ; s2 = n + sum (n - i) b_i  (mod 65521)
// Each block reduces a 64 KiB tile to (sum, weighted sum); the host folds the per-tile pairs (a few
// integers per 64 KiB -- framing arithmetic, not a pass over the data).
// ---------------------------------------------------------------------------------------------
constexpr uint32_t ADLER_TILE = 1u << 16;
__global__ void __launch_bounds__(256) k_adler_tiles(const uint8_t *__restrict__ p, size_t n, uint64_t *__restrict__ part) {
  const size_t base = (size_t)blockIdx.x * ADLER_TILE;
  const uint32_t len = (uint32_t)min((size_t)ADLER_TILE, n - base);
  uint64_t s = 0, ws = 0;  // ws = sum (len - i) * b_i  within the tile
  for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) {
    uint32_t b = p[base + i];
    s += b;
    ws += (uint64_t)(len - i) * b;
  }
  __shared__ uint64_t sh[2][8];
  for (int d = 16; d >= 1; d >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, d);
    ws += __shfl_xor_sync(0xffffffffu, ws, d);
  }
  if ((threadIdx.x & 31) == 0) {
    sh[0][threadIdx.x >> 5] = s;
    sh[1][threadIdx.x >> 5] = ws;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint64_t a = 0, b = 0;
    for (int i = 0; i < 8; ++i) {
      a += sh[0][i];
      b += sh[1][i];
    }
    part[2 * blockIdx.x] = a;
    part[2 * blockIdx.x + 1] = b;
  }
}

// device buffer -> adler32 (blocking)
static int device_adler32(const uint8_t *d, size_t n, uint32_t *out) {
  const uint32_t MOD = 65521;
  if (n == 0) {
    *out = 1;
    return B200Z_OK;
  }
  size_t tiles = (n + ADLER_TILE - 1) / ADLER_TILE;
  CU(g.d_small.reserve(tiles * 16));
  k_adler_tiles<<<(unsigned)tiles, 256, 0, g.stream>>>(d, n, (uint64_t *)g.d_small.p);
  count_launch();
  CU(cudaGetLastError());
  std::vector<uint64_t> part(tiles * 2);
  CU(cudaMemcpyAsync(part.data(), g.d_small.p, tiles * 16, cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  uint64_t s1 = 1, s2 = 0;
  for (size_t t = 0; t < tiles; ++t) {
    uint64_t len = (t + 1 == tiles) ? n - t * ADLER_TILE : ADLER_TILE;
    uint64_t ts = part[2 * t] % MOD, tw = part[2 * t + 1] % MOD;
    // appending a tile: s2' = s2 + len * s1 + tw ; s1' = s1 + ts
    s2 = (s2 + (len % MOD) * s1 + tw) % MOD;
    s1 = (s1 + ts) % MOD;
  }
  *out = (uint32_t)((s2 << 16) | s1);
  return B200Z_OK;
}

// ---------------------------------------------------------------------------------------------
// batch plumbing
// ---------------------------------------------------------------------------------------------
struct MetaLayout {
  size_t n;
  size_t off_in_off, off_out_off, off_in_len, off_out_cap, off_out_len, off_status, off_in_used, bytes;
  explicit MetaLayout(size_t n_) : n(n_) {
    size_t o = 0;
    off_in_off = o;
    o += 8 * n;
    off_out_off = o;
    o += 8 * n;
    off_in_len = o;
    o += 4 * n;
    off_out_cap = o;
    o += 4 * n;
    off_out_len = o;
    o += 4 * n;
    off_status = o;
    o += 4 * n;
    off_in_used = o;
    o += 4 * n;
    bytes = align_up(o, 256);
  }
  size_t inputs_bytes() const { return off_out_len; }
};

static size_t workspace_bytes(size_t n_units, size_t total_out_cap) { return inflate_ws_bytes(n_units, total_out_cap); }

// Runs one batch whose compressed bytes are ALREADY in g.d_in (at offset 0 = in_base) and whose
// output goes to g.d_out.  Meta arrays are host arrays; results are copied back into them.
static int run_batch_on_staged(const uint64_t *in_off, const uint32_t *in_len, const uint64_t *out_off,
                               const uint32_t *out_cap, uint32_t *out_len, int32_t *status, uint32_t *in_used,
                               size_t n, size_t out_extent, bool count_only = false, uint32_t hist = 0) {
  MetaLayout ml(n);
  CU(g.h_meta.reserve(ml.bytes));
  CU(g.d_meta.reserve(ml.bytes));
  uint8_t *hm = (uint8_t *)g.h_meta.p;
  memcpy(hm + ml.off_in_off, in_off, 8 * n);
  memcpy(hm + ml.off_out_off, out_off, 8 * n);
  memcpy(hm + ml.off_in_len, in_len, 4 * n);
  memcpy(hm + ml.off_out_cap, out_cap, 4 * n);
  CU(cudaMemcpyAsync(g.d_meta.p, hm, ml.inputs_bytes(), cudaMemcpyHostToDevice, g.stream));
  const size_t ws = workspace_bytes(n, out_extent);
  CU(g.d_ws.reserve(ws));
  uint8_t *dm = (uint8_t *)g.d_meta.p;
  InflateBatch b;
  b.in_base = (const uint8_t *)g.d_in.p;
  b.in_off = (const uint64_t *)(dm + ml.off_in_off);
  b.in_len = (const uint32_t *)(dm + ml.off_in_len);
  b.out_base = (uint8_t *)g.d_out.p;
  b.out_off = (const uint64_t *)(dm + ml.off_out_off);
  b.out_cap = (const uint32_t *)(dm + ml.off_out_cap);
  b.out_len = (uint32_t *)(dm + ml.off_out_len);
  b.status = (int32_t *)(dm + ml.off_status);
  b.in_used = (uint32_t *)(dm + ml.off_in_used);
  b.n_units = n;
  b.ws = inflate_ws_carve(g.d_ws.p, n, out_extent);
  b.ws.hist = hist;
  b.count_only = count_only;
  CU(launch_inflate(b, g.stream));
  CU(cudaMemcpyAsync(hm + ml.off_out_len, dm + ml.off_out_len, ml.bytes - ml.off_out_len, cudaMemcpyDeviceToHost,
                     g.stream));
  CU(cudaStreamSynchronize(g.stream));
  memcpy(out_len, hm + ml.off_out_len, 4 * n);
  memcpy(status, hm + ml.off_status, 4 * n);
  memcpy(in_used, hm + ml.off_in_used, 4 * n);
  return B200Z_OK;
}

cudaError_t copy_slots_to_host(uint8_t *host, const uint8_t *dev, uint64_t lo, const uint64_t *out_off, const uint32_t *out_cap,
                               size_t n, cudaStream_t stream) {
  std::vector<std::pair<uint64_t, uint64_t>> slots;
  slots.reserve(n);
  for (size_t u = 0; u < n; ++u)
    if (out_cap[u]) slots.emplace_back(out_off[u], out_off[u] + out_cap[u]);
  std::sort(slots.begin(), slots.end());
  size_t i = 0;
  while (i < slots.size()) {
    const uint64_t a = slots[i].first;
    uint64_t b = slots[i].second;
    for (++i; i < slots.size() && slots[i].first <= b; ++i) b = std::max(b, slots[i].second);
    const cudaError_t e = cudaMemcpyAsync(host + a, dev + (a - lo), b - a, cudaMemcpyDeviceToHost, stream);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

static int stage_input(const uint8_t *in, size_t n) {
  CU(g.d_in.reserve(n + 64));
  if (n) CU(cudaMemcpyAsync(g.d_in.p, in, n, cudaMemcpyHostToDevice, g.stream));
  return B200Z_OK;
}

// largest possible DEFLATE expansion: a 258-byte match costs at least 2 bits
static size_t max_inflate_out(size_t in_len) {
  const size_t lim = (size_t)0xffffffffu;
  if (in_len > lim / 1040) return lim;
  return in_len * 1040 + 1024;
}

// one stream from staged input at [pos, in_total): returns unit results
struct OneResult {
  uint32_t out_len, in_used;
  int32_t status;
};
// `shared_output`: the stream is a gzip member -- everything already in g.d_out[0, out_pos) belongs to the same OutputStream
// and is within reach of its back-references (InflateWs::hist)
static int run_one_staged(size_t pos, size_t in_total, size_t out_pos, size_t out_cap_total, OneResult *r,
                          bool shared_output = false) {
  uint64_t io = pos, oo = out_pos;
  size_t avail_in = in_total - pos;
  uint32_t il = (uint32_t)(avail_in > 0xfffffff0u ? 0xfffffff0u : avail_in);
  size_t room = out_cap_total - out_pos;
  size_t mx = max_inflate_out(il);
  if (room > mx) room = mx;
  uint32_t oc = (uint32_t)(room > 0xfffffff0u ? 0xfffffff0u : room);
  CU(g.d_out.reserve_keep(out_pos + oc + 64, out_pos, g.stream));
  const uint32_t hist = shared_output ? (uint32_t)(out_pos > 65535 ? 65535 : out_pos) : 0u;  // distances end at 32768
  return run_batch_on_staged(&io, &il, &oo, &oc, &r->out_len, &r->status, &r->in_used, 1, out_pos + oc, false, hist);
}

static inline uint32_t le32(const uint8_t *p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }
static inline uint32_t le16(const uint8_t *p) { return p[0] | (p[1] << 8); }

// _readHeader (_gzip_decoder_web.dart:60-138).  Returns 1 ok, 0 "not gzip" (-> zlib fallback), -1 = the
// Dart code would have thrown (readByte past the end).  *bsize = BGZF 'BC' member size hint or 0.
static int gzip_header(const uint8_t *in, size_t n, size_t pos, size_t *hdr_end, size_t *bsize) {
  *bsize = 0;
  if (pos + 2 > n) return -1;
  if (le16(in + pos) != 0x8b1f) return 0;
  if (pos + 3 > n) return -1;
  if (in[pos + 2] != 8) return 0;
  if (pos + 10 > n) return -1;
  uint8_t flags = in[pos + 3];
  size_t p = pos + 10;
  if (flags & 0x04) {
    if (p + 2 > n) return -1;
    size_t xlen = le16(in + p);
    p += 2;
    size_t xend = p + xlen;
    if (xend > n) xend = n;  // readBytes clamps (input_stream.dart:132-136)
    // look for the BGZF subfield  'B' 'C' SLEN=2  BSIZE(u16) = member size - 1
    size_t q = p;
    while (q + 4 <= xend) {
      size_t slen = le16(in + q + 2);
      if (in[q] == 'B' && in[q + 1] == 'C' && slen == 2 && q + 6 <= xend) *bsize = (size_t)le16(in + q + 4) + 1;
      q += 4 + slen;
    }
    p = xend;
  }
  if (flags & 0x08) {
    while (p < n && in[p] != 0) ++p;
    if (p < n) ++p;
  }
  if (flags & 0x10) {
    while (p < n && in[p] != 0) ++p;
    if (p < n) ++p;
  }
  if (flags & 0x02) {
    if (p + 2 > n) return -1;
    p += 2;
  }
  *hdr_end = p;
  return 1;
}

static int zlib_decode_staged(const uint8_t *in, size_t in_len, size_t pos, int verify, int raw, int big_endian,
                              size_t out_pos, size_t out_cap, size_t *out_len_total);

// An ISIZE that DEFLATE cannot reach from `comp` bytes (1032:1 at most: a 258-byte match costs two bits) is no size hint:
// such a member is decoded the hint-free way instead of being believed (it would size buffers).
static inline bool isize_possible(uint32_t isize, size_t comp) { return (uint64_t)isize <= (uint64_t)comp * 1040u + 1024u; }

// THE definition of a hinted run: whole members from `pos` on that carry the BGZF 'BC' size and a believable ISIZE.
// Returns the position behind the run; appends the members to `ms` when given; *out_bytes = what their ISIZE fields promise.
// (struct HintedMember: b200z_internal.h)
static size_t hinted_run(const uint8_t *in, size_t n, size_t pos, std::vector<HintedMember> *ms, size_t *out_bytes) {
  size_t p = pos, o = 0;
  while (p < n) {
    size_t hdr_end, bsize;
    if (gzip_header(in, n, p, &hdr_end, &bsize) != 1 || bsize == 0) break;
    const size_t next = p + bsize;
    if (next > n || next < hdr_end + 8) break;
    const uint32_t isize = le32(in + next - 4);
    if (!isize_possible(isize, next - hdr_end)) break;
    if (ms) ms->push_back({hdr_end, next, isize});
    o += isize;
    p = next;
  }
  if (out_bytes) *out_bytes = o;
  return p;
}

// GZip member loop on staged input.
static int gzip_decode_staged(const uint8_t *in, size_t in_len, int verify, size_t out_cap, size_t *out_len_total,
                              size_t pos = 0, size_t out_pos = 0) {
  std::vector<uint64_t> v_in_off, v_out_off;
  std::vector<uint32_t> v_in_len, v_out_cap, v_out_len, v_in_used;
  std::vector<int32_t> v_status;
  std::vector<size_t> v_next;
  while (pos < in_len) {
    // -------- gather a run of members that carry a size hint (BGZF 'BC' + ISIZE) --------
    v_in_off.clear(); v_out_off.clear(); v_in_len.clear(); v_out_cap.clear(); v_next.clear();
    size_t o = out_pos;
    {
      std::vector<HintedMember> run;
      hinted_run(in, in_len, pos, &run, nullptr);
      for (const HintedMember &m : run) {
        v_in_off.push_back(m.hdr_end);
        v_in_len.push_back((uint32_t)(m.next - m.hdr_end));
        v_out_off.push_back(o);
        v_out_cap.push_back(m.isize);
        v_next.push_back(m.next);
        o += m.isize;
      }
    }
    size_t nb = v_in_off.size();
    if (nb > 0) {
      if (o > out_cap) {
        *out_len_total = o;  // best knowledge of what is needed so far
        set_err("gzip_decode: output needs at least %zu bytes, out_cap %zu", o, out_cap);
        return B200Z_E_NOSPC;
      }
      CU(g.d_out.reserve_keep(o + 64, out_pos, g.stream));
      v_out_len.resize(nb); v_status.resize(nb); v_in_used.resize(nb);
      int rc = run_batch_on_staged(v_in_off.data(), v_in_len.data(), v_out_off.data(), v_out_cap.data(),
                                   v_out_len.data(), v_status.data(), v_in_used.data(), nb, o);
      if (rc) return rc;
      // accept the prefix whose hints were exact; anything else is redone the slow, hint-free way
      size_t k = 0;
      for (; k < nb; ++k) {
        bool ok = v_status[k] == B200Z_U_DONE && v_out_len[k] == v_out_cap[k] &&
                  (size_t)v_in_off[k] + v_in_used[k] + 8 == v_next[k];
        if (!ok) break;
      }
      if (k > 0) {
        pos = v_next[k - 1];
        out_pos = v_out_off[k - 1] + v_out_len[k - 1];
      }
      if (k == nb) continue;
    }
    if (pos >= in_len) break;
    // -------- one member without (valid) hints: decode it alone to learn where it ends --------
    size_t hdr_end, bsize;
    int h = gzip_header(in, in_len, pos, &hdr_end, &bsize);
    if (h < 0) {
      *out_len_total = out_pos;
      set_err("gzip_decode: truncated header (Dart: RangeError)");
      return B200Z_E_THROW;
    }
    if (h == 0)  // no gzip header: fall back to zlib on the same little-endian stream (:31-37)
      return zlib_decode_staged(in, in_len, pos, verify & B200Z_GZIP_VERIFY, (verify & B200Z_GZIP_RAW) != 0, /*big_endian=*/0, out_pos,
                                out_cap, out_len_total);  // decodeStream(input, output, verify: verify, raw: raw)
    OneResult r;
    int rc = run_one_staged(hdr_end, in_len, out_pos, out_cap, &r, /*shared_output=*/true);
    if (rc) return rc;
    out_pos += r.out_len;
    *out_len_total = out_pos;
    if (r.status == B200Z_U_NOSPC) {
      set_err("gzip_decode: out_cap %zu too small", out_cap);
      return B200Z_E_NOSPC;
    }
    if (r.status == B200Z_U_RANGE || r.status == B200Z_U_THROW) {
      set_err("gzip_decode: member at %zu: Dart would throw RangeError (status %d)", pos, r.status);
      return B200Z_E_THROW;
    }
    size_t after = hdr_end + r.in_used;
    if (r.status == B200Z_U_STOP && after + 8 > in_len) {
      // Inflate gave up because the input ran out inside a block (inflate.dart:166-168, 192-195): the byte-wise bit reader
      // has pulled every byte by then, so the two readUint32 of the trailer (:40-41) start past the end -- RangeError.
      // This is what a truncated file does.
      set_err("gzip_decode: member at %zu: input ends inside the stream (Dart: RangeError)", pos);
      return B200Z_E_THROW;
    }
    if (r.status != B200Z_U_DONE && r.status != B200Z_U_EOS) {
      set_err("gzip_decode: member at %zu stopped with status %d", pos, r.status);
      return B200Z_E_DATA;  // DESIGN.md "Divergences": reference keeps parsing from an unspecified position
    }
    if (after + 8 > in_len) {  // readUint32 x2 past the end (:40-41)
      set_err("gzip_decode: truncated trailer (Dart: RangeError)");
      return B200Z_E_THROW;
    }
    pos = after + 8;
  }
  *out_len_total = out_pos;
  return B200Z_OK;
}


// ---------------------------------------------------------------------------------------------
// End-to-end fast path for the common shape: a run of members that all carry size hints.  The run is cut
// into chunks; chunk c's host->device copy, its two kernels and chunk c-1's device->host copy run on
// three streams, so the PCIe transfers hide behind each other and behind the decode.  Every hint is
// verified afterwards; the first member whose hint was not exact ends the accepted prefix and the
// caller continues from there on the slow, hint-free path (same bytes out either way).
// ---------------------------------------------------------------------------------------------
static int gzip_fast_path_piped_fwd(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap, size_t *pos_io, size_t *out_pos_io,
                                    size_t *needed);
static int gzip_fast_path(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap, size_t *pos_io,
                          size_t *out_pos_io, size_t *needed) {
  // B200Z_GZIP_PIPED_WALK=1: the walk inside the pipeline (below).  Off by default: measured on a B200 (config 2, pinned
  // buffers) it is SLOWER, 34.9 ms per call against 24.0 ms for walk-first -- see the comment on gzip_fast_path_piped.
  {
    const char *pe = getenv("B200Z_GZIP_PIPED_WALK");
    const bool piped = pe && atoi(pe) != 0;
    const size_t span = in_len - *pos_io, room = out_cap >= *out_pos_io ? out_cap - *out_pos_io : 0;
    if (piped && *pos_io < in_len && room <= 32 * span + (64u << 20)) return gzip_fast_path_piped_fwd(in, in_len, out, out_cap, pos_io, out_pos_io, needed);
  }
  std::vector<HintedMember> ms;
  size_t promised = 0;
  const size_t p = hinted_run(in, in_len, *pos_io, &ms, &promised);
  const size_t o = *out_pos_io + promised;
  const size_t nb = ms.size();
  if (nb == 0) return B200Z_OK;
  if (o > out_cap) {
    *needed = o;
    set_err("gzip_decode: output needs at least %zu bytes, out_cap %zu", o, out_cap);
    return B200Z_E_NOSPC;
  }
  const size_t in_lo = *pos_io, in_hi = p, out_lo = *out_pos_io;
  // chunks: ~8 per call (one compute stream each, so their kernels overlap: a stream's decode time is set by
  // its token count, not by how many streams run beside it), at least 4 MiB of compressed bytes each
  size_t min_chunk = 4u << 20;  // (B200Z_GZIP_CHUNK_KB: smaller chunks for tests of the pipeline itself)
  if (const char *e = getenv("B200Z_GZIP_CHUNK_KB")) min_chunk = std::max<size_t>(1, (size_t)atoll(e)) << 10;
  size_t target = (in_hi - in_lo) / Ctx::kCompStreams;
  if (target < min_chunk) target = min_chunk;
  // The device->host copy of the output bounds this path (it moves ~2.5x the bytes of the input copy over the same link),
  // and it cannot start before the first chunk has been copied in and decoded: the first two chunks are a quarter and a
  // half of a regular one, so that it starts early and is fed without a gap from then on.  (B200Z_GZIP_RAMP=0: equal chunks.)
  const char *ramp_env = getenv("B200Z_GZIP_RAMP");
  const bool ramp = !ramp_env || atoi(ramp_env) != 0;
  std::vector<size_t> cut{0};
  {
    size_t acc_start = in_lo;
    for (size_t i = 0; i < nb; ++i) {
      size_t want = target;
      if (ramp && cut.size() <= 2) want = std::max<size_t>(target >> (3 - cut.size()), min_chunk);  // chunk 0: /4, chunk 1: /2
      if (ms[i].next - acc_start >= want && i + 1 < nb) {
        cut.push_back(i + 1);
        acc_start = ms[i].next;
      }
    }
    cut.push_back(nb);
  }
  const size_t nchunks = cut.size() - 1;
  MetaLayout ml(nb);
  CU(g.h_meta.reserve(ml.bytes));
  CU(g.d_meta.reserve(ml.bytes));
  CU(g.d_in.reserve(in_len + 64));
  CU(g.d_out.reserve_keep(o + 64, out_lo, g.stream));
  uint8_t *hm = (uint8_t *)g.h_meta.p, *dm = (uint8_t *)g.d_meta.p;
  uint64_t *h_in_off = (uint64_t *)(hm + ml.off_in_off), *h_out_off = (uint64_t *)(hm + ml.off_out_off);
  uint32_t *h_in_len = (uint32_t *)(hm + ml.off_in_len), *h_out_cap = (uint32_t *)(hm + ml.off_out_cap);
  size_t max_chunk_out = 0;
  std::vector<size_t> chunk_out_lo(nchunks + 1);
  {
    size_t oo = out_lo;
    for (size_t c = 0; c < nchunks; ++c) {
      chunk_out_lo[c] = oo;
      size_t rel = 0;
      for (size_t i = cut[c]; i < cut[c + 1]; ++i) {
        h_in_off[i] = ms[i].hdr_end;
        h_in_len[i] = (uint32_t)(ms[i].next - ms[i].hdr_end);
        h_out_off[i] = rel;  // relative to the chunk's slice of d_out
        h_out_cap[i] = ms[i].isize;
        rel += ms[i].isize;
      }
      oo += rel;
      if (rel > max_chunk_out) max_chunk_out = rel;
    }
    chunk_out_lo[nchunks] = oo;
  }
  size_t max_units = 0;
  for (size_t c = 0; c < nchunks; ++c) max_units = cut[c + 1] - cut[c] > max_units ? cut[c + 1] - cut[c] : max_units;
  (void)max_units;
  (void)max_chunk_out;
  CU(g.d_ws.reserve(inflate_ws_bytes(nb, o - out_lo)));  // token layout mirrors the output layout
  const InflateWs ws_all = inflate_ws_carve(g.d_ws.p, nb, o - out_lo);
  std::vector<cudaEvent_t> ev_in(nchunks), ev_k(nchunks);
  for (size_t c = 0; c < nchunks; ++c) {
    CU(cudaEventCreateWithFlags(&ev_in[c], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&ev_k[c], cudaEventDisableTiming));
  }
  CU(cudaMemcpyAsync(dm, hm, ml.inputs_bytes(), cudaMemcpyHostToDevice, g.s_h2d));
  int rc = B200Z_OK;
  for (size_t c = 0; c < nchunks && rc == B200Z_OK; ++c) {
    const size_t a = cut[c], b = cut[c + 1];
    const size_t lo = c == 0 ? in_lo : ms[a - 1].next, hi = ms[b - 1].next;
    CU(cudaMemcpyAsync((uint8_t *)g.d_in.p + lo, in + lo, hi - lo, cudaMemcpyHostToDevice, g.s_h2d));
    CU(cudaEventRecord(ev_in[c], g.s_h2d));
    cudaStream_t cs = g.s_comp[c % Ctx::kCompStreams];
    CU(cudaStreamWaitEvent(cs, ev_in[c], 0));
    InflateBatch bt;
    bt.in_base = (const uint8_t *)g.d_in.p;
    bt.in_off = (const uint64_t *)(dm + ml.off_in_off) + a;
    bt.in_len = (const uint32_t *)(dm + ml.off_in_len) + a;
    bt.out_base = (uint8_t *)g.d_out.p + chunk_out_lo[c];
    bt.out_off = (const uint64_t *)(dm + ml.off_out_off) + a;
    bt.out_cap = (const uint32_t *)(dm + ml.off_out_cap) + a;
    bt.out_len = (uint32_t *)(dm + ml.off_out_len) + a;
    bt.status = (int32_t *)(dm + ml.off_status) + a;
    bt.in_used = (uint32_t *)(dm + ml.off_in_used) + a;
    bt.n_units = b - a;
    bt.share = (int)(nchunks < (size_t)Ctx::kCompStreams ? nchunks : (size_t)Ctx::kCompStreams);
    bt.ws = inflate_ws_slice(ws_all, a, chunk_out_lo[c] - out_lo);
    CU(launch_inflate(bt, cs));
    CU(cudaEventRecord(ev_k[c], cs));
    CU(cudaStreamWaitEvent(g.s_d2h, ev_k[c], 0));
    const size_t ob = chunk_out_lo[c + 1] - chunk_out_lo[c];
    if (ob) CU(cudaMemcpyAsync(out + chunk_out_lo[c], (uint8_t *)g.d_out.p + chunk_out_lo[c], ob, cudaMemcpyDeviceToHost, g.s_d2h));
  }
  CU(cudaMemcpyAsync(hm + ml.off_out_len, dm + ml.off_out_len, ml.bytes - ml.off_out_len, cudaMemcpyDeviceToHost, g.s_d2h));
  CU(cudaStreamSynchronize(g.s_d2h));
  for (size_t c = 0; c < nchunks; ++c) {
    cudaEventDestroy(ev_in[c]);
    cudaEventDestroy(ev_k[c]);
  }
  const uint32_t *r_len = (const uint32_t *)(hm + ml.off_out_len), *r_used = (const uint32_t *)(hm + ml.off_in_used);
  const int32_t *r_st = (const int32_t *)(hm + ml.off_status);
  size_t k = 0;
  for (; k < nb; ++k) {
    bool ok = r_st[k] == B200Z_U_DONE && r_len[k] == ms[k].isize && ms[k].hdr_end + r_used[k] + 8 == ms[k].next;
    if (!ok) break;
  }
  if (k > 0) {
    *pos_io = ms[k - 1].next;
    size_t oo = out_lo;
    for (size_t i = 0; i < k; ++i) oo += ms[i].isize;
    *out_pos_io = oo;
  }
  return B200Z_OK;
}

// ---------------------------------------------------------------------------------------------
// The same path with the HOST walk inside the pipeline.  Finding the members is a pointer chase through the compressed
// bytes (a member's size is in its own header): 0.35 us per member, 5.7 ms for the 16 384 members of a GiB -- a fifth of
// the whole call when it runs before anything else starts.  Here every chunk is sent and launched as soon as the walk
// has covered its members, and the walk of the next chunk runs while the device works on this one.  Buffers are sized
// from what the caller offers (out_cap) instead of from the walk's totals, so this form is taken when that is a sane
// bound; anything unexpected (a hint that overflows out_cap, more members than the tables were sized for) ends the run
// early and the caller goes on from the returned position exactly as before.
// MEASURED (round 2, B200, config 2): 34.9 ms per call, against 24.0 ms with the walk in front -- in both forms tried
// (whole input sent ahead in 16 MiB pieces; one copy per chunk as here).  The walk is a chain of dependent cache misses
// into the caller's buffer, and it now runs while the copy engines move 100 GB/s through the same host memory; the
// chunks reach the device later than the device could take them.  Kept as an option (B200Z_GZIP_PIPED_WALK=1) with its
// tests; the default is walk-first.
// ---------------------------------------------------------------------------------------------
static int gzip_fast_path_piped(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap, size_t *pos_io, size_t *out_pos_io,
                                size_t *needed) {
  const size_t in_lo = *pos_io, out_lo = *out_pos_io;
  size_t hdr0, bsize0;
  if (in_lo >= in_len || gzip_header(in, in_len, in_lo, &hdr0, &bsize0) != 1 || bsize0 == 0) return B200Z_OK;
  const size_t room = out_cap - out_lo;
  const size_t span = in_len - in_lo;
  // members expected: from the first one's size, with slack; the tables are sized once
  size_t nb_cap = span / bsize0;
  nb_cap = nb_cap + nb_cap / 4 + 4096;
  size_t min_chunk = 4u << 20;
  if (const char *e = getenv("B200Z_GZIP_CHUNK_KB")) min_chunk = std::max<size_t>(1, (size_t)atoll(e)) << 10;
  size_t target = span / Ctx::kCompStreams;
  if (target < min_chunk) target = min_chunk;
  const char *ramp_env = getenv("B200Z_GZIP_RAMP");
  const bool ramp = !ramp_env || atoi(ramp_env) != 0;

  MetaLayout ml(nb_cap);
  CU(g.h_meta.reserve(ml.bytes));
  CU(g.d_meta.reserve(ml.bytes));
  CU(g.d_in.reserve(in_len + 64));
  CU(g.d_out.reserve_keep(out_lo + room + 64, out_lo, g.stream));
  CU(g.d_ws.reserve(inflate_ws_bytes(nb_cap, room)));
  const InflateWs ws_all = inflate_ws_carve(g.d_ws.p, nb_cap, room);
  uint8_t *hm = (uint8_t *)g.h_meta.p, *dm = (uint8_t *)g.d_meta.p;
  uint64_t *h_in_off = (uint64_t *)(hm + ml.off_in_off), *h_out_off = (uint64_t *)(hm + ml.off_out_off);
  uint32_t *h_in_len = (uint32_t *)(hm + ml.off_in_len), *h_out_cap = (uint32_t *)(hm + ml.off_out_cap);

  std::vector<cudaEvent_t> ev_k, ev_piece;
  std::vector<HintedMember> ms;
  ms.reserve(nb_cap);
  size_t p = in_lo, o = out_lo;          // walk position, output position
  size_t chunk_a = 0, chunk_in_lo = in_lo, chunk_out_lo = out_lo, n_chunks = 0;
  bool nospc = false;
  auto launch_chunk = [&](size_t a, size_t b) -> int {  // members [a, b): bytes [chunk_in_lo, ms[b-1].next) -> [chunk_out_lo, o)
    const size_t hi = ms[b - 1].next;
    cudaStream_t cs = g.s_comp[n_chunks % Ctx::kCompStreams];
    // the chunk's bytes, then (on the chunk's stream, behind them on the copy engine) its slices of the four input arrays.
    // (Sending the whole input ahead in one go was tried: the small copies below then queue behind ALL of it on the
    // host-to-device engine and the first decode starts 7 ms late -- 34.8 ms per call instead of 24.3.)
    cudaEvent_t ei;
    CU(cudaEventCreateWithFlags(&ei, cudaEventDisableTiming));
    ev_piece.push_back(ei);
    CU(cudaMemcpyAsync((uint8_t *)g.d_in.p + chunk_in_lo, in + chunk_in_lo, hi - chunk_in_lo, cudaMemcpyHostToDevice, g.s_h2d));
    CU(cudaEventRecord(ei, g.s_h2d));
    CU(cudaStreamWaitEvent(cs, ei, 0));
    CU(cudaMemcpyAsync(dm + ml.off_in_off + 8 * a, hm + ml.off_in_off + 8 * a, 8 * (b - a), cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(dm + ml.off_out_off + 8 * a, hm + ml.off_out_off + 8 * a, 8 * (b - a), cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(dm + ml.off_in_len + 4 * a, hm + ml.off_in_len + 4 * a, 4 * (b - a), cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpyAsync(dm + ml.off_out_cap + 4 * a, hm + ml.off_out_cap + 4 * a, 4 * (b - a), cudaMemcpyHostToDevice, cs));
    InflateBatch bt;
    bt.in_base = (const uint8_t *)g.d_in.p;
    bt.in_off = (const uint64_t *)(dm + ml.off_in_off) + a;
    bt.in_len = (const uint32_t *)(dm + ml.off_in_len) + a;
    bt.out_base = (uint8_t *)g.d_out.p + chunk_out_lo;
    bt.out_off = (const uint64_t *)(dm + ml.off_out_off) + a;
    bt.out_cap = (const uint32_t *)(dm + ml.off_out_cap) + a;
    bt.out_len = (uint32_t *)(dm + ml.off_out_len) + a;
    bt.status = (int32_t *)(dm + ml.off_status) + a;
    bt.in_used = (uint32_t *)(dm + ml.off_in_used) + a;
    bt.n_units = b - a;
    bt.share = Ctx::kCompStreams;
    bt.ws = inflate_ws_slice(ws_all, a, chunk_out_lo - out_lo);
    CU(launch_inflate(bt, cs));
    cudaEvent_t ek;
    CU(cudaEventCreateWithFlags(&ek, cudaEventDisableTiming));
    ev_k.push_back(ek);
    CU(cudaEventRecord(ek, cs));
    CU(cudaStreamWaitEvent(g.s_d2h, ek, 0));
    const size_t ob = o - chunk_out_lo;
    if (ob) CU(cudaMemcpyAsync(out + chunk_out_lo, (uint8_t *)g.d_out.p + chunk_out_lo, ob, cudaMemcpyDeviceToHost, g.s_d2h));
    n_chunks++;
    chunk_a = b;
    chunk_in_lo = hi;
    chunk_out_lo = o;
    return B200Z_OK;
  };
  int rc = B200Z_OK;
  size_t promised = out_lo;  // what the hints ask for, also beyond out_cap (reported with B200Z_E_NOSPC)
  while (p < in_len && ms.size() < nb_cap) {
    size_t hdr_end, bsize;
    if (gzip_header(in, in_len, p, &hdr_end, &bsize) != 1 || bsize == 0) break;
    const size_t next = p + bsize;
    if (next > in_len || next < hdr_end + 8) break;
    const uint32_t isize = le32(in + next - 4);
    if (!isize_possible(isize, next - hdr_end)) break;
    promised += isize;
    if (promised > out_cap) nospc = true;
    if (!nospc) {
      const size_t i = ms.size();
      ms.push_back({hdr_end, next, isize});
      h_in_off[i] = hdr_end;
      h_in_len[i] = (uint32_t)(next - hdr_end);
      h_out_off[i] = o - chunk_out_lo;  // relative to the chunk's slice of d_out
      h_out_cap[i] = isize;
      o += isize;
      size_t want = target;
      if (ramp && n_chunks < 2) want = std::max<size_t>(target >> (2 - n_chunks), min_chunk);  // chunk 0: /4, chunk 1: /2
      if (next - chunk_in_lo >= want) {
        rc = launch_chunk(chunk_a, ms.size());
        if (rc) break;
      }
    }
    p = next;
  }
  if (rc == B200Z_OK && !nospc && chunk_a < ms.size()) rc = launch_chunk(chunk_a, ms.size());
  const size_t nb = ms.size();
  if (rc == B200Z_OK && nb) {
    CU(cudaMemcpyAsync(hm + ml.off_out_len, dm + ml.off_out_len, 4 * nb, cudaMemcpyDeviceToHost, g.s_d2h));
    CU(cudaMemcpyAsync(hm + ml.off_status, dm + ml.off_status, 4 * nb, cudaMemcpyDeviceToHost, g.s_d2h));
    CU(cudaMemcpyAsync(hm + ml.off_in_used, dm + ml.off_in_used, 4 * nb, cudaMemcpyDeviceToHost, g.s_d2h));
  }
  CU(cudaStreamSynchronize(g.s_h2d));
  CU(cudaStreamSynchronize(g.s_d2h));
  for (cudaEvent_t e : ev_piece) cudaEventDestroy(e);
  for (cudaEvent_t e : ev_k) cudaEventDestroy(e);
  if (rc) return rc;
  if (nospc) {
    *needed = promised;
    set_err("gzip_decode: output needs at least %zu bytes, out_cap %zu", promised, out_cap);
    return B200Z_E_NOSPC;
  }
  const uint32_t *r_len = (const uint32_t *)(hm + ml.off_out_len), *r_used = (const uint32_t *)(hm + ml.off_in_used);
  const int32_t *r_st = (const int32_t *)(hm + ml.off_status);
  size_t k = 0, oo = out_lo;
  for (; k < nb; ++k) {
    const bool ok = r_st[k] == B200Z_U_DONE && r_len[k] == ms[k].isize && ms[k].hdr_end + r_used[k] + 8 == ms[k].next;
    if (!ok) break;
    oo += ms[k].isize;
  }
  if (k > 0) {
    *pos_io = ms[k - 1].next;
    *out_pos_io = oo;
  }
  return B200Z_OK;
}

static int gzip_fast_path_piped_fwd(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap, size_t *pos_io, size_t *out_pos_io,
                                    size_t *needed) {
  return gzip_fast_path_piped(in, in_len, out, out_cap, pos_io, out_pos_io, needed);
}

// ---- hooks for the file-stream layer (b200z_file.cu) ----
void set_error_text(const char *msg) { set_err("%s", msg); }

// Bytes of `in` covered by whole members that carry a size hint, from offset 0 (the run gzip_fast_path would take), and the
// output bytes their ISIZE fields promise.
size_t gzip_hinted_prefix(const uint8_t *in, size_t n, size_t *out_bytes) { return hinted_run(in, n, 0, nullptr, out_bytes); }
size_t gzip_hinted_members(const uint8_t *in, size_t n, size_t pos, std::vector<HintedMember> *ms, size_t *out_bytes) {
  return hinted_run(in, n, pos, ms, out_bytes);
}

// The hinted run at the front of `in`, decoded through the chunk pipeline: *in_used = end of the last member whose hint
// was exact (== the whole run unless a hint lied), *out_len = the bytes those members produced.
int gzip_decode_hinted(const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *in_used, size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  size_t pos = 0, out_pos = 0, needed = 0;
  rc = gzip_fast_path(in, n, out, out_cap, &pos, &out_pos, &needed);
  *in_used = pos;
  *out_len = rc == B200Z_E_NOSPC ? needed : out_pos;
  return rc;
}

// The member loop over `in`, continuing a decodeStream call that has already produced output: its last `hist_len` bytes
// (<= 65535; distances end at 32768) are placed in front, because the members share one OutputStream and may copy from it
// (InflateWs::hist).  *out_len counts the new bytes only.
int gzip_decode_after(const uint8_t *in, size_t n, int verify, const uint8_t *hist, size_t hist_len, uint8_t *out, size_t out_cap,
                      size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  rc = stage_input(in, n);
  if (rc) return rc;
  CU(g.d_out.reserve(hist_len + 64));
  if (hist_len) CU(cudaMemcpyAsync(g.d_out.p, hist, hist_len, cudaMemcpyHostToDevice, g.stream));
  size_t total = hist_len;
  rc = gzip_decode_staged(in, n, verify, out_cap + hist_len, &total, 0, hist_len);
  const size_t produced = total > hist_len ? total - hist_len : 0;
  *out_len = produced;
  if (rc == B200Z_E_NOSPC || rc == B200Z_E_NODEVICE) return rc;
  const size_t hi = produced > out_cap ? out_cap : produced;
  if (hi) CU(cudaMemcpyAsync(out, (const uint8_t *)g.d_out.p + hist_len, hi, cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  return rc;
}

// _zlib_decoder_web.dart:31-107 on staged input.
static int zlib_decode_staged(const uint8_t *in, size_t in_len, size_t pos, int verify, int raw, int big_endian,
                              size_t out_pos, size_t out_cap, size_t *out_len_total) {
  // The reference inflates every stream into a buffer of its own and hands it to `output` only when the NEXT stream's
  // header has been accepted, or at the end of the loop (:82-84, :101-103).  A stream whose successor's header is bad, or
  // whose Adler-32 is wrong or missing, therefore never reaches the output.  Here the streams are decoded straight into
  // their final position; `committed` is what `output` holds, `pending` the bytes of the stream that waits.
  size_t committed = out_pos, pending = 0;
  *out_len_total = committed;
  while (pos < in_len) {
    if (!raw) {
      if (pos + 2 > in_len) {
        set_err("zlib_decode: truncated header (Dart: RangeError)");
        return B200Z_E_THROW;
      }
      uint32_t cmf = in[pos], flg = in[pos + 1];
      pos += 2;
      if ((cmf & 8) != 8) {  // :57 (sic)
        set_err("zlib_decode: method != deflate");
        return B200Z_E_DATA;
      }
      if (((cmf * 256) + flg) % 31 != 0) {
        set_err("zlib_decode: bad FCHECK");
        return B200Z_E_DATA;
      }
      if ((flg & 32) != 0) {
        if (pos + 4 > in_len) {
          set_err("zlib_decode: truncated DICTID (Dart: RangeError)");
          return B200Z_E_THROW;
        }
        set_err("zlib_decode: FDICT not supported");
        return B200Z_E_DATA;
      }
    }
    committed += pending;  // output.writeBytes(buffer) (:82-84)
    pending = 0;
    *out_len_total = committed;
    OneResult r;
    int rc = run_one_staged(pos, in_len, committed, out_cap, &r);
    if (rc) return rc;
    if (r.status == B200Z_U_NOSPC) {
      *out_len_total = committed + r.out_len;
      set_err("zlib_decode: out_cap %zu too small", out_cap);
      return B200Z_E_NOSPC;
    }
    if (r.status == B200Z_U_RANGE || r.status == B200Z_U_THROW) {
      set_err("zlib_decode: Dart would throw RangeError (status %d)", r.status);
      return B200Z_E_THROW;
    }
    if (r.status == B200Z_U_BADCODE) {
      *out_len_total = committed + r.out_len;
      set_err("zlib_decode: unusable Huffman code set");
      return B200Z_E_DATA;
    }
    pos += r.in_used;
    if (r.status == B200Z_U_STOP && pos < in_len) {
      // Inflate gave up with input left: the reference's stream position is then wherever its byte-wise bit buffer had
      // got to (not rewound) -- unspecified; stop here with the partial output (DESIGN.md "Divergences").
      *out_len_total = committed + r.out_len;
      set_err("zlib_decode: inflate stopped early");
      return B200Z_E_DATA;
    }
    // (B200Z_U_STOP with the input used up == the stream ends inside a block: Inflate simply returns what it has, :85)
    if (!raw) {
      if (pos + 4 > in_len) {  // readUint32 past the end (:88); the stream's bytes were not handed over yet
        set_err("zlib_decode: truncated Adler-32 (Dart: RangeError)");
        return B200Z_E_THROW;
      }
      uint32_t stored = big_endian ? ((uint32_t)in[pos] << 24 | in[pos + 1] << 16 | in[pos + 2] << 8 | in[pos + 3])
                                   : le32(in + pos);
      pos += 4;
      if (verify) {
        uint32_t a;
        rc = device_adler32((const uint8_t *)g.d_out.p + committed, r.out_len, &a);
        if (rc) return rc;
        if (a != stored) {
          set_err("zlib_decode: Adler-32 mismatch");
          return B200Z_E_DATA;  // this stream's bytes are dropped (:91-94)
        }
      }
    }
    pending = r.out_len;
  }
  *out_len_total = committed + pending;  // (:101-103)
  return B200Z_OK;
}

}  // namespace b200z


// =============================================================================================
// BZip2Decoder.decodeBytes / decodeStream  (bzip2_decoder.dart:13-88)
// Host side: stream header, ordering + chain validation of the block candidates the scan kernel finds,
// stored-CRC comparison.  All bit/byte work is in bzip2_kernels.cu.
// =============================================================================================
namespace b200z {

struct Carver {  // carve typed arrays out of one device allocation
  uint8_t *p;
  size_t off = 0;
  explicit Carver(void *base) : p((uint8_t *)base) {}
  template <typename T>
  T *take(size_t n) {
    off = align_up(off, 256);
    T *r = p ? (T *)(p + off) : nullptr;
    off += n * sizeof(T);
    return r;
  }
};

static inline uint32_t be32_at_bit(const uint8_t *in, size_t n, uint64_t bit) {
  uint64_t v = 0;
  size_t b0 = (size_t)(bit >> 3);
  for (int i = 0; i < 5; ++i) v = (v << 8) | (b0 + i < n ? in[b0 + i] : 0);
  return (uint32_t)(v >> (8 - (bit & 7)));
}

// shard != nullptr: decode only this rank's share of the block candidates and report every block instead of walking the
// chain (the ranks' reports are merged and validated by the caller, archive_b200/shard.py).
struct Bz2Shard {
  uint32_t rank, world;
  b200z_bz2_block *blocks;
  size_t blocks_cap, n_blocks;
};
static int bzip2_decode_impl(const uint8_t *in, size_t in_len, int verify, uint8_t *out, size_t out_cap, size_t *out_len,
                             Bz2Shard *shard = nullptr) {
  *out_len = 0;
  // 'B' 'Z' 'h' level: each is a readByte() that throws at EOS (bz2_bit_reader.dart:17-20)
  static const uint8_t sig[3] = {0x42, 0x5a, 0x68};
  for (int i = 0; i < 3; ++i) {
    if ((size_t)i >= in_len) {
      set_err("bzip2: truncated signature (Dart: RangeError)");
      return B200Z_E_THROW;
    }
    if (in[i] != sig[i]) {
      set_err("bzip2: bad signature");
      return B200Z_E_DATA;
    }
  }
  if (in_len < 4) {
    set_err("bzip2: truncated header (Dart: RangeError)");
    return B200Z_E_THROW;
  }
  const int level = (int)in[3] - 0x30;
  if (level < 0 || level > 9) {
    set_err("bzip2: bad block size");
    return B200Z_E_DATA;
  }
  if (in_len == 4) return B200Z_OK;  // while (!input.isEOS) never runs
  const uint32_t nblock_max = (uint32_t)level * 100000u;
  const uint64_t total_bits = (uint64_t)in_len * 8;

  int rc = stage_input(in, in_len);
  if (rc) return rc;
  CU(cudaMemsetAsync((uint8_t *)g.d_in.p + in_len, 0, 64, g.stream));

  // ---- K6: candidates ----
  const uint32_t cand_cap = 1u << 20;
  CU(g.d_small.reserve((size_t)cand_cap * 8 + 256));
  unsigned long long *d_cand = (unsigned long long *)((uint8_t *)g.d_small.p + 256);
  uint32_t *d_ncand = (uint32_t *)g.d_small.p;
  CU(bz2_launch_scan((const uint8_t *)g.d_in.p, in_len, d_cand, d_ncand, cand_cap, g.stream));
  uint32_t ncand = 0;
  CU(cudaMemcpyAsync(&ncand, d_ncand, 4, cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  if (ncand > cand_cap) {
    set_err("bzip2: more than %u magic candidates", cand_cap);
    return B200Z_E_INTERNAL;
  }
  std::vector<unsigned long long> cand(ncand);
  if (ncand) CU(cudaMemcpy(cand.data(), d_cand, (size_t)ncand * 8, cudaMemcpyDeviceToHost));
  std::sort(cand.begin(), cand.end(), [](unsigned long long a, unsigned long long b) {
    return (a & ~(1ull << 63)) < (b & ~(1ull << 63));
  });
  std::vector<unsigned long long> blk_bits;
  std::vector<uint32_t> blk_of_cand(ncand, 0xffffffffu);
  for (uint32_t i = 0; i < ncand; ++i)
    if (!(cand[i] >> 63)) {
      blk_of_cand[i] = (uint32_t)blk_bits.size();
      blk_bits.push_back(cand[i]);
    }
  const uint32_t nb = (uint32_t)blk_bits.size();

  // ---- device arrays ----
  const uint32_t chunks_max = (nblock_max + 1023) / 1024;
  const uint32_t nb_all = nb ? nb : 1;
  auto carve = [&](void *base, uint32_t nbk) {
    Carver c(base);
    struct A {
      unsigned long long *blk_bit, *end_bit, *block_out, *block_off;
      uint32_t *rec_val, *rec_pos, *n_rec, *nblock, *orig_ptr, *rnd, *chist, *tt, *seg_len, *seg_next, *seg_off, *seg_resume, *slice_state,
          *slice_out, *block_crc, *cycle_len, *fast, *walk_ctr;
      int32_t *status, *irregular;
      uint8_t *sym8, *raw, *slots;
      BzChainHost *chain;
      size_t bytes;
    } a;
    a.blk_bit = c.take<unsigned long long>(nb_all);
    a.end_bit = c.take<unsigned long long>(nbk);
    a.block_out = c.take<unsigned long long>(nbk);
    a.block_off = c.take<unsigned long long>(nbk + 1);
    a.n_rec = c.take<uint32_t>(nbk);
    a.nblock = c.take<uint32_t>(nbk);
    a.orig_ptr = c.take<uint32_t>(nbk);
    a.rnd = c.take<uint32_t>(nbk);
    a.status = c.take<int32_t>(nbk);
    a.irregular = c.take<int32_t>(nbk);
    a.block_crc = c.take<uint32_t>(nbk);
    a.cycle_len = c.take<uint32_t>(nbk);
    a.fast = c.take<uint32_t>(nbk);
    a.walk_ctr = c.take<uint32_t>(4);
    a.chain = c.take<BzChainHost>(nbk);
    a.seg_len = c.take<uint32_t>((size_t)nbk * 4098);
    a.seg_next = c.take<uint32_t>((size_t)nbk * 4098);
    a.seg_off = c.take<uint32_t>((size_t)nbk * 4098);
    a.seg_resume = c.take<uint32_t>((size_t)nbk * 4098);
    a.slice_state = c.take<uint32_t>((size_t)nbk * 1024);
    a.slice_out = c.take<uint32_t>((size_t)nbk * 1024);
    a.chist = c.take<uint32_t>((size_t)nbk * chunks_max * 256);
    a.rec_val = c.take<uint32_t>((size_t)nbk * nblock_max);
    a.rec_pos = c.take<uint32_t>((size_t)nbk * nblock_max);
    a.tt = c.take<uint32_t>((size_t)nbk * nblock_max);
    a.sym8 = c.take<uint8_t>((size_t)nbk * nblock_max);
    a.raw = c.take<uint8_t>((size_t)nbk * nblock_max);
    a.slots = c.take<uint8_t>((size_t)nbk * bz2_slot_bytes_per_block());
    a.bytes = align_up(c.off, 256);
    return a;
  };
  uint32_t nbk = nb ? nb : 1;
  if (shard) {  // only this rank's share needs the big per-block arrays (blk_bit keeps all candidates: small)
    const uint32_t lo = (uint32_t)((uint64_t)nb * shard->rank / shard->world), hi = (uint32_t)((uint64_t)nb * (shard->rank + 1) / shard->world);
    nbk = hi > lo ? hi - lo : 1;
  }
  auto sz = carve(nullptr, nbk);
  CU(g.d_bz.reserve(sz.bytes));
  auto A = carve(g.d_bz.p, nbk);

  // ---- K7 on every candidate (speculative: a magic-looking bit pattern inside a block just decodes to junk) ----
  std::vector<uint32_t> h_nrec(nb), h_nblock(nb), h_optr(nb), h_rnd(nb);
  std::vector<unsigned long long> h_end(nb);
  std::vector<int32_t> h_st(nb);
  uint32_t k_lo = 0, k_hi = nb;  // candidates this call decodes
  if (shard) {
    k_lo = (uint32_t)((uint64_t)nb * shard->rank / shard->world);
    k_hi = (uint32_t)((uint64_t)nb * (shard->rank + 1) / shard->world);
  }
  if (k_hi > k_lo) {
    CU(cudaMemcpyAsync(A.blk_bit, blk_bits.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, g.stream));
    Bz2Entropy e;
    e.words = (const uint32_t *)g.d_in.p;
    e.n_bytes = in_len;
    e.blk_bit = A.blk_bit + k_lo;
    e.n_blocks = k_hi - k_lo;
    e.nblock_max = nblock_max;
    // block k of this call uses slot k - k_lo of every per-block array
    e.rec_val = A.rec_val; e.rec_pos = A.rec_pos; e.n_rec = A.n_rec; e.nblock = A.nblock; e.orig_ptr = A.orig_ptr;
    e.randomised = A.rnd; e.end_bit = A.end_bit; e.status = A.status; e.fast_flag = A.fast; e.sym8 = A.sym8;
    CU(bz2_launch_entropy(e, g.stream));
    const uint32_t m = k_hi - k_lo;
    auto fetch = [&]() -> int {
      CU(cudaMemcpyAsync(h_nrec.data() + k_lo, A.n_rec, m * 4, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaMemcpyAsync(h_nblock.data() + k_lo, A.nblock, m * 4, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaMemcpyAsync(h_optr.data() + k_lo, A.orig_ptr, m * 4, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaMemcpyAsync(h_rnd.data() + k_lo, A.rnd, m * 4, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaMemcpyAsync(h_end.data() + k_lo, A.end_bit, (size_t)m * 8, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaMemcpyAsync(h_st.data() + k_lo, A.status, m * 4, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaStreamSynchronize(g.stream));
      return B200Z_OK;
    };
    rc = fetch();
    if (rc) return rc;
    {
      std::vector<uint32_t> h_fast(m);
      CU(cudaMemcpy(h_fast.data(), A.fast, (size_t)m * 4, cudaMemcpyDeviceToHost));
      unsigned long long nf = 0;
      for (uint32_t v : h_fast) nf += v;
      g_bz2_fast_blocks += nf;
      g_bz2_exact_blocks += m - nf;
    }
    // damaged blocks that the reference keeps decoding past a bad Huffman code (K7 status -3): decoded again the reference's
    // way, one thread each (bzip2_kernels.cu: k_bz2_entropy_literal); intact streams have none
    std::vector<uint32_t> quirk;
    for (uint32_t k = k_lo; k < k_hi; ++k)
      if (h_st[k] == -3) quirk.push_back(k - k_lo);
    if (!quirk.empty()) {
      uint32_t *d_list = (uint32_t *)((uint8_t *)g.d_small.p + 256);  // the candidate list is on the host by now
      CU(cudaMemcpyAsync(d_list, quirk.data(), quirk.size() * 4, cudaMemcpyHostToDevice, g.stream));
      CU(bz2_launch_entropy_literal(e, d_list, (uint32_t)quirk.size(), g.stream));
      rc = fetch();
      if (rc) return rc;
    }
  }

  // ---- walk the chain exactly as decodeStream's loop does (:46-87) ----
  std::vector<BzChainHost> chain;
  std::vector<uint32_t> stored_crc;
  int final_rc = B200Z_OK;
  bool have_eos = false;
  uint32_t eos_crc = 0;
  uint64_t pos = 32;
  size_t ci = 0;
  std::vector<uint32_t> chain_of(nb, 0xffffffffu);
  if (shard) {
    for (uint32_t k = k_lo; k < k_hi; ++k)
      if (h_st[k] == 0) {
        chain_of[k] = (uint32_t)chain.size();
        chain.push_back({k - k_lo, h_nblock[k], h_nrec[k], h_optr[k], h_rnd[k] ? 1u : 0u});
        stored_crc.push_back(blk_bits[k] + 80 <= total_bits ? be32_at_bit(in, in_len, blk_bits[k] + 48) : 0u);
      }
  }
  for (; !shard;) {
    if ((pos + 7) / 8 >= in_len) break;  // input.isEOS: every byte has been pulled into the bit reader
    if (pos + 48 > total_bits) {
      // _readBlockType (:90-111) reads its 6 bytes one at a time: the first one that fits neither magic returns -1 before
      // the missing bytes are asked for (RangeError)
      static const uint8_t blk_magic[6] = {0x31, 0x41, 0x59, 0x26, 0x53, 0x59}, eos_magic[6] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90};
      bool blk = true, eos = true, mismatch = false;
      for (int i = 0; i < 6 && pos + 8 * (uint64_t)(i + 1) <= total_bits; ++i) {
        const uint8_t b = (uint8_t)(be32_at_bit(in, in_len, pos + 8 * (uint64_t)i) >> 24);
        blk = blk && b == blk_magic[i];
        eos = eos && b == eos_magic[i];
        if (!blk && !eos) {
          mismatch = true;
          break;
        }
      }
      if (mismatch) {
        set_err("bzip2: no block signature at bit %llu", (unsigned long long)pos);
        final_rc = B200Z_E_DATA;
      } else {
        set_err("bzip2: truncated block header (Dart: RangeError)");
        final_rc = B200Z_E_THROW;
      }
      break;
    }
    while (ci < ncand && (cand[ci] & ~(1ull << 63)) < pos) ++ci;
    if (ci >= ncand || (cand[ci] & ~(1ull << 63)) != pos) {
      set_err("bzip2: no block signature at bit %llu", (unsigned long long)pos);
      final_rc = B200Z_E_DATA;  // _readBlockType -> -1 -> false
      break;
    }
    if (pos + 80 > total_bits) {  // 4 CRC bytes follow either magic
      set_err("bzip2: truncated CRC (Dart: RangeError)");
      final_rc = B200Z_E_THROW;
      break;
    }
    const uint32_t crc_field = be32_at_bit(in, in_len, pos + 48);
    if (cand[ci] >> 63) {
      have_eos = true;
      eos_crc = crc_field;
      break;  // end of stream: whatever follows is ignored (:83-84)
    }
    const uint32_t k = blk_of_cand[ci];
    if (h_st[k] == -2) {
      set_err("bzip2: block at bit %llu reads past the end (Dart: RangeError)", (unsigned long long)pos);
      final_rc = B200Z_E_THROW;
      break;
    }
    if (h_st[k] != 0) {
      set_err("bzip2: data error in the block at bit %llu", (unsigned long long)pos);
      final_rc = B200Z_E_DATA;
      break;
    }
    chain.push_back({k, h_nblock[k], h_nrec[k], h_optr[k], h_rnd[k] ? 1u : 0u});  // randomised blocks: serial walk in K8
    stored_crc.push_back(crc_field);
    pos = h_end[k];
  }

  if (getenv("B200Z_DEBUG")) {
    fprintf(stderr, "[b200z] bzip2: %u candidates (%u block), chain %zu, rc so far %d, eos %d\n", ncand, nb, chain.size(),
            final_rc, (int)have_eos);
    for (uint32_t i = 0; i < nb && i < 16; ++i)
      fprintf(stderr, "[b200z]   cand %u bit %llu st %d nblock %u nrec %u optr %u end %llu\n", i,
              (unsigned long long)blk_bits[i], h_st[i], h_nblock[i], h_nrec[i], h_optr[i], (unsigned long long)h_end[i]);
  }
  // ---- K8 on the chain ----
  const uint32_t nc = (uint32_t)chain.size();
  std::vector<unsigned long long> h_off(nc + 1, 0);
  size_t early_copied = 0;  // bytes [0, early_copied) of the output are on their way to the host already (s_d2h)
  std::vector<uint32_t> h_crc(nc);
  std::vector<int32_t> h_irr(nc);
  if (nc) {
    CU(g.d_out.reserve(out_cap + 64));
    CU(cudaMemcpyAsync(A.chain, chain.data(), (size_t)nc * sizeof(BzChainHost), cudaMemcpyHostToDevice, g.stream));
    Bz2Ibwt w;
    w.chain = A.chain; w.n_chain = nc; w.nblock_max = nblock_max;
    w.rec_val = A.rec_val; w.rec_pos = A.rec_pos; w.sym8 = A.sym8; w.chist = A.chist; w.tt = A.tt;
    w.seg_len = A.seg_len; w.seg_next = A.seg_next; w.seg_off = A.seg_off; w.seg_resume = A.seg_resume; w.slots = A.slots; w.walk_ctr = A.walk_ctr; w.irregular = A.irregular; w.cycle_len = A.cycle_len; w.raw = A.raw;
    w.slice_state = A.slice_state; w.slice_out = A.slice_out; w.block_out = A.block_out; w.block_off = A.block_off;
    w.block_crc = A.block_crc; w.out = (uint8_t *)g.d_out.p; w.out_cap = out_cap;
    for (const BzChainHost &ce : chain) w.any_randomised = w.any_randomised || (ce.flags & 1u);
    w.any_records = false;
    for (const BzChainHost &ce : chain) w.any_records = w.any_records || ce.n_rec != 0;
    // B200Z_BZ2_GROUPS=n decodes a long chain in n groups, the bytes of a finished group on their way to the host (copy
    // stream) while the next group is decoded.  Measured on a B200 (512 MiB, 597 blocks): 59.4 ms in one piece, 64.5 ms in
    // 4 groups, 73.8 ms in 8 -- the pointer-chasing kernels of K8 are bound by latency, not by the number of blocks, so a
    // group costs nearly what the whole chain costs.  Off by default.
    uint32_t groups = 1u;
    if (const char *ge = getenv("B200Z_BZ2_GROUPS")) groups = (uint32_t)std::max(1, atoi(ge));
    if (shard || groups > nc) groups = 1;
    // The RLE1 output pass (per block, 3.5 ms for 597 blocks) runs in 4 groups and a finished group's bytes go to the host on
    // the copy stream while the next group is written: the blocks' offsets are known before it, so nothing waits
    // (B200Z_BZ2_EMIT_GROUPS, 1: one pass, one copy at the end).
    uint32_t emit_groups = (!shard && nc >= 64) ? 4u : 1u;
    if (const char *ge = getenv("B200Z_BZ2_EMIT_GROUPS")) emit_groups = (uint32_t)std::max(1, atoi(ge));
    if (shard || emit_groups > nc || groups > 1) emit_groups = 1;
    if (groups <= 1 && emit_groups > 1) {
      w.phase = 1;
      CU(bz2_launch_ibwt(w, g.stream));
      CU(cudaMemcpyAsync(h_off.data(), A.block_off, (size_t)(nc + 1) * 8, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaStreamSynchronize(g.stream));
      w.phase = 2;
      for (uint32_t gi = 0; gi < emit_groups; ++gi) {
        const uint32_t lo = (uint32_t)((uint64_t)nc * gi / emit_groups), hi = (uint32_t)((uint64_t)nc * (gi + 1) / emit_groups);
        CU(bz2_launch_ibwt_group(w, lo, hi, g.stream));
        cudaEvent_t ev;
        CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        CU(cudaEventRecord(ev, g.stream));
        CU(cudaStreamWaitEvent(g.s_d2h, ev, 0));
        cudaEventDestroy(ev);  // (released once it has completed)
        const size_t end = (size_t)(h_off[hi] < (unsigned long long)out_cap ? h_off[hi] : (unsigned long long)out_cap);
        if (end > early_copied) {
          CU(cudaMemcpyAsync(out + early_copied, (uint8_t *)g.d_out.p + early_copied, end - early_copied, cudaMemcpyDeviceToHost,
                             g.s_d2h));
          early_copied = end;
        }
      }
      w.phase = 0;
    } else if (groups <= 1) {
      CU(bz2_launch_ibwt(w, g.stream));
    } else {
      CU(g.h_meta.reserve((size_t)groups * 8));
      volatile unsigned long long *h_end_off = (volatile unsigned long long *)g.h_meta.p;
      std::vector<cudaEvent_t> ev(groups);
      for (uint32_t gi = 0; gi < groups; ++gi) {
        const uint32_t lo = (uint32_t)((uint64_t)nc * gi / groups), hi = (uint32_t)((uint64_t)nc * (gi + 1) / groups);
        CU(bz2_launch_ibwt_group(w, lo, hi, g.stream));
        CU(cudaMemcpyAsync((void *)(h_end_off + gi), A.block_off + hi, 8, cudaMemcpyDeviceToHost, g.stream));
        CU(cudaEventCreateWithFlags(&ev[gi], cudaEventDisableTiming));
        CU(cudaEventRecord(ev[gi], g.stream));
      }
      for (uint32_t gi = 0; gi < groups; ++gi) {
        CU(cudaEventSynchronize(ev[gi]));
        cudaEventDestroy(ev[gi]);
        const unsigned long long eo = h_end_off[gi];
        const size_t end = (size_t)(eo < (unsigned long long)out_cap ? eo : (unsigned long long)out_cap);
        if (end > early_copied) {
          CU(cudaMemcpyAsync(out + early_copied, (uint8_t *)g.d_out.p + early_copied, end - early_copied, cudaMemcpyDeviceToHost,
                             g.s_d2h));
          early_copied = end;
        }
      }
    }
    CU(cudaMemcpyAsync(h_off.data(), A.block_off, (size_t)(nc + 1) * 8, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaMemcpyAsync(h_crc.data(), A.block_crc, (size_t)nc * 4, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaMemcpyAsync(h_irr.data(), A.irregular, (size_t)nc * 4, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    if (early_copied) CU(cudaStreamSynchronize(g.s_d2h));  // (no copy into the caller's buffer outlives this call)
  }
  if (getenv("B200Z_DEBUG"))
    for (uint32_t i = 0; i < nc && i < 16; ++i)
      fprintf(stderr, "[b200z]   chain %u off %llu..%llu crc %08x stored %08x irregular %d\n", i, (unsigned long long)h_off[i],
              (unsigned long long)h_off[i + 1], h_crc[i], stored_crc[i], h_irr[i]);
  if (shard) {
    // one report per candidate of the range + one per end-of-stream candidate (every rank reports those)
    shard->n_blocks = 0;
    auto push = [&](const b200z_bz2_block &b) {
      if (shard->n_blocks < shard->blocks_cap) shard->blocks[shard->n_blocks] = b;
      shard->n_blocks++;
    };
    for (uint32_t k = k_lo; k < k_hi; ++k) {
      b200z_bz2_block b{};
      b.start_bit = blk_bits[k];
      b.end_bit = h_end[k];
      b.status = h_st[k];
      b.flags = 0u;  // randomised blocks are decoded like the others (serial walk)
      b.crc_stored = blk_bits[k] + 80 <= total_bits ? be32_at_bit(in, in_len, blk_bits[k] + 48) : 0u;
      const uint32_t c = chain_of[k];
      if (c != 0xffffffffu) {
        b.out_bytes = h_off[c + 1] - h_off[c];
        b.crc_calc = h_crc[c];
        if (h_irr[c] == 2) b.flags |= B200Z_BZ2_OVERRUN;
        else if (h_irr[c]) b.flags |= B200Z_BZ2_CORRUPT_CYCLE;
      }
      push(b);
    }
    for (uint32_t i = 0; i < ncand; ++i)
      if (cand[i] >> 63) {
        b200z_bz2_block b{};
        b.start_bit = cand[i] & ~(1ull << 63);
        b.end_bit = b.start_bit + 80;
        b.flags = B200Z_BZ2_EOS;
        b.crc_stored = b.start_bit + 80 <= total_bits ? be32_at_bit(in, in_len, b.start_bit + 48) : 0u;
        push(b);
      }
    const size_t n_local = nc ? (size_t)h_off[nc] : 0;
    *out_len = n_local;
    if (shard->n_blocks > shard->blocks_cap) {
      set_err("bzip2 shard: %zu block reports, capacity %zu", shard->n_blocks, shard->blocks_cap);
      return B200Z_E_NOSPC;
    }
    if (n_local > out_cap) {
      set_err("bzip2 shard: output needs %zu bytes, out_cap %zu", n_local, out_cap);
      return B200Z_E_NOSPC;
    }
    if (n_local) CU(cudaMemcpyAsync(out, g.d_out.p, n_local, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    return B200Z_OK;
  }
  // blocks are committed in order; the first bad one ends the stream (its bytes are already written when the
  // reference compares the CRC, :58-66)
  size_t n_out = 0;
  uint32_t combined = 0;
  for (uint32_t i = 0; i < nc; ++i) {
    if (h_irr[i] == 1) {
      set_err("bzip2: block %u: corrupt BWT cycle", i);
      final_rc = B200Z_E_DATA;
      break;
    }
    n_out = (size_t)h_off[i + 1];
    if (h_irr[i] == 2) {  // the run-length walk overran the block (:497-499, :628-631): false, its bytes are already written
      set_err("bzip2: block %u: run overruns the block", i);
      final_rc = B200Z_E_DATA;
      have_eos = false;
      break;
    }
    if (verify && h_crc[i] != stored_crc[i]) {
      set_err("bzip2: block %u CRC mismatch", i);
      final_rc = B200Z_E_DATA;
      have_eos = false;
      break;
    }
    combined = ((combined << 1) | (combined >> 31)) ^ h_crc[i];
  }
  if (final_rc == B200Z_OK && have_eos && verify && eos_crc != combined) {
    set_err("bzip2: combined CRC mismatch");
    final_rc = B200Z_E_DATA;
  }
  *out_len = n_out;
  if (n_out > out_cap) {
    set_err("bzip2: output needs %zu bytes, out_cap %zu", n_out, out_cap);
    return B200Z_E_NOSPC;
  }
  if (n_out > early_copied)
    CU(cudaMemcpyAsync(out + early_copied, (uint8_t *)g.d_out.p + early_copied, n_out - early_copied, cudaMemcpyDeviceToHost,
                       g.stream));
  CU(cudaStreamSynchronize(g.stream));
  return final_rc;
}

}  // namespace b200z

// =============================================================================================
// Deflate(bytes, level:, windowBits:).getBytes() + crc32  (deflate.dart:25-100), and the encoder framing of
// _zlib_encoder_web.dart:27-73 / _gzip_encoder_web.dart:27-100
// =============================================================================================
namespace b200z {

// CRC-32 (reflected 0xEDB88320) combination, as in zlib's crc32_combine: crc(A||B) = crc(A) * x^(8|B|) + crc(B)
static uint32_t crc_multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}
static uint32_t crc_xpow8(uint64_t nbytes) {
  uint32_t p = 1u << 31;      // x^0
  uint32_t sq = 1u << 23;     // x^8 in the reflected representation (bit 31 = x^0)
  while (nbytes) {
    if (nbytes & 1) p = crc_multmodp(sq, p);
    sq = crc_multmodp(sq, sq);
    nbytes >>= 1;
  }
  return p;
}
static const uint32_t kCrcTile = 1u << 13;
// CRC-32 of d[0, n) on stream s: tile CRCs into d_part ((n / kCrcTile + 1) words of device memory), folded on the host
static int device_crc32_on(const uint8_t *d, size_t n, uint32_t *d_part, cudaStream_t s, uint32_t *out) {
  const uint32_t TILE = kCrcTile;
  if (n == 0) {
    *out = 0;
    return B200Z_OK;
  }
  size_t tiles = (n + TILE - 1) / TILE;
  CU(crc32_tiles_device(d, n, TILE, d_part, s));
  std::vector<uint32_t> part(tiles);
  CU(cudaMemcpyAsync(part.data(), d_part, tiles * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  uint32_t crc = part[0];
  const uint32_t xfull = crc_xpow8(TILE);
  for (size_t t = 1; t < tiles; ++t) {
    size_t len = (t + 1 == tiles) ? n - t * TILE : TILE;
    crc = crc_multmodp(len == TILE ? xfull : crc_xpow8(len), crc) ^ part[t];
  }
  *out = crc;
  return B200Z_OK;
}
static int device_crc32(const uint8_t *d, size_t n, uint32_t *out) {
  CU(g.d_small.reserve((n / kCrcTile + 1) * 4 + 256));
  return device_crc32_on(d, n, (uint32_t *)g.d_small.p, g.stream, out);
}

// the old deflate_stored (deflate.dart:691-737) touches no data: its block list follows from the length alone
// windowBits sets the window (deflate.dart:132-134) and with it where the blocks are cut: 2^windowBits - 262 bytes at most
static void stored_block_list(size_t n, int window_bits, std::vector<DeflStoredBlock> &out) {
  const long long w_size = 1ll << window_bits, window_size = 2 * w_size, min_lookahead = 262;
  const long long max_block_size = 65536 - 5 < 0xffff ? 65536 - 5 : 0xffff;
  long long strstart = 0, block_start = 0, lookahead = 0, base = 0;  // base: absolute position of window index 0
  long long in_pos = 0;
  auto flush = [&](bool eof) {
    // (block_start is never negative here: a block is flushed once it is w_size - min_lookahead long, and the window
    // slides only when strstart has reached 2 * w_size - min_lookahead, so the data is always still there to be stored)
    out.push_back({(uint32_t)(base + block_start), (uint32_t)(strstart - block_start), eof ? 1u : 0u});
    block_start = strstart;
  };
  auto fill_window = [&]() {
    do {
      long long more = window_size - lookahead - strstart;
      if (more == 0 && strstart == 0 && lookahead == 0) {
        more = w_size;
      } else if (strstart >= w_size + w_size - min_lookahead) {
        strstart -= w_size;
        block_start -= w_size;
        base += w_size;
        more += w_size;
      }
      if (in_pos >= (long long)n) return;
      long long len = (long long)n - in_pos;
      if (len > more) len = more;
      in_pos += len;
      lookahead += len;
    } while (lookahead < min_lookahead && in_pos < (long long)n);
  };
  for (;;) {
    if (lookahead <= 1) {
      fill_window();
      if (lookahead == 0) break;
    }
    strstart += lookahead;
    lookahead = 0;
    const long long max_start = block_start + max_block_size;
    if (strstart >= max_start) {
      lookahead = strstart - max_start;
      strstart = max_start;
      flush(false);
    }
    if (strstart - block_start >= w_size - min_lookahead) flush(false);
  }
  flush(true);
}

// compresses d_in[0, n) (already staged in g.d_in) into g.d_out; returns the compressed size
static int deflate_staged(size_t n, int level, int window_bits, size_t *out_len) {
  if (window_bits < 9 || window_bits > 15 || level < 0 || level > 9) {
    set_err("deflate: invalid level %d / windowBits %d (Dart: LateInitializationError)", level, window_bits);
    return B200Z_E_ARG;
  }
  if (n >= 0xffff0000ull) {
    set_err("deflate: inputs of 4 GiB and more are not supported");
    return B200Z_E_ARG;
  }
  const size_t cap = align_up(deflate_bound(n) + 16, 256);
  CU(g.d_out.reserve(cap));
  if (level == 0) {
    std::vector<DeflStoredBlock> bl;
    stored_block_list(n, window_bits, bl);
    const size_t ws = bl.size() * 64 + 1024;
    CU(g.d_ws.reserve(ws));
    CU(deflate_stored_device((const uint8_t *)g.d_in.p, bl.data(), (uint32_t)bl.size(), (uint8_t *)g.d_out.p, cap, g.d_ws.p,
                             g.d_ws.cap, out_len, g.stream));
    return B200Z_OK;
  }
  const size_t ws = deflate_workspace_bytes(n);
  CU(g.d_ws.reserve(ws));
  uint32_t stats[3];
  CU(deflate_slow_device((const uint8_t *)g.d_in.p, n, level, window_bits, (uint8_t *)g.d_out.p, cap, g.d_ws.p, g.d_ws.cap, out_len, stats,
                         g.stream));
  return B200Z_OK;
}

// ---------------------------------------------------------------------------------------------
// Many independent streams at once (ZipEncoder's members, zip_encoder.dart:185-259).  One stream's kernels are a chain
// with three host round trips (token count, block count, bit count) and, at levels 1-3, a single serial thread: a lone
// member leaves the device almost idle.  All inputs are staged with one burst of copies; `lanes` host threads then take
// members off a counter, each with its own CUDA stream, workspace and output slot, so the chains of different members
// overlap on the device.  Every member is compressed exactly as b200z_deflate_raw compresses it.
// ---------------------------------------------------------------------------------------------
static int deflate_member_on(const uint8_t *d_in, size_t n, int level, int window_bits, uint8_t *d_out, size_t cap, void *ws,
                             size_t ws_bytes, cudaStream_t s, size_t *out_len, uint32_t *crc, const DeflFastMember *pre = nullptr) {
  if (level == 0) {
    std::vector<DeflStoredBlock> bl;
    stored_block_list(n, window_bits, bl);
    CU(deflate_stored_device(d_in, bl.data(), (uint32_t)bl.size(), d_out, cap, ws, ws_bytes, out_len, s));
  } else {
    uint32_t stats[3];
    CU(deflate_slow_device(d_in, n, level, window_bits, d_out, cap, ws, ws_bytes, out_len, stats, s, pre));
  }
  // the tile CRCs go to the front of the workspace: the encoder is done with it (both paths end synchronised)
  return device_crc32_on(d_in, n, (uint32_t *)ws, s, crc);
}

static int deflate_batch_impl(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len, size_t n_units, int level,
                              int window_bits, uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                              uint64_t *out_len, uint32_t *crc32, int32_t *status) {
  std::vector<size_t> din(n_units + 1), dout(n_units + 1);
  size_t ws_lane = 4096, acc_in = 0, acc_out = 0;
  for (size_t i = 0; i < n_units; ++i) {
    const size_t n = (size_t)in_len[i];
    if (n >= 0xffff0000ull) {
      set_err("deflate_batch: unit %zu: inputs of 4 GiB and more are not supported", i);
      return B200Z_E_ARG;
    }
    din[i] = acc_in;
    dout[i] = acc_out;
    acc_in += align_up(n + 64, 256);
    acc_out += align_up(deflate_bound(n) + 16, 256);
    size_t ws = (n / kCrcTile + 1) * 4 + 256;
    if (level == 0) {
      std::vector<DeflStoredBlock> bl;
      stored_block_list(n, window_bits, bl);
      ws = std::max(ws, bl.size() * 64 + 1024);
    } else {
      ws = std::max(ws, deflate_workspace_bytes(n));
    }
    ws_lane = std::max(ws_lane, align_up(ws, 256));
  }
  din[n_units] = acc_in;
  dout[n_units] = acc_out;
  size_t lanes = Ctx::kCompStreams;
  if (const char *e = getenv("B200Z_DEFLATE_LANES")) lanes = (size_t)atoi(e);
  lanes = std::max<size_t>(1, std::min<size_t>(std::min<size_t>(lanes, Ctx::kCompStreams), n_units));
  CU(g.d_in.reserve(acc_in + 64));
  CU(g.d_out.reserve(acc_out + 64));
  CU(g.d_ws.reserve(lanes * ws_lane));
  cudaEvent_t staged;
  CU(cudaEventCreateWithFlags(&staged, cudaEventDisableTiming));
  CU(cudaMemsetAsync(g.d_in.p, 0, acc_in, g.s_h2d));  // the bytes behind every member read as zeros (as in deflate_raw)
  for (size_t i = 0; i < n_units; ++i)
    if (in_len[i])
      CU(cudaMemcpyAsync((uint8_t *)g.d_in.p + din[i], in_base + in_off[i], (size_t)in_len[i], cudaMemcpyHostToDevice, g.s_h2d));
  CU(cudaEventRecord(staged, g.s_h2d));
  std::atomic<size_t> next{0};
  size_t next_end = n_units;  // the lanes take members [next, next_end)
  std::vector<int> lane_rc(lanes, B200Z_OK);
  std::vector<std::string> lane_err(lanes);
  std::vector<DeflFastMember> pre;  // levels 1-3: where the batch kernel has put every member's tokens
  const int device = g.device;
  auto lane = [&](size_t l) {
    auto fail = [&](int rc) {
      lane_rc[l] = rc;
      lane_err[l] = t_err;
      next.store(n_units);  // the other lanes stop taking members
    };
    if (cudaSetDevice(device) != cudaSuccess) return fail(B200Z_E_NODEVICE);  // a new thread starts on device 0
    cudaStream_t s = g.s_comp[l];
    if (cudaStreamWaitEvent(s, staged, 0) != cudaSuccess) return fail(B200Z_E_NODEVICE);
    void *ws = (uint8_t *)g.d_ws.p + l * ws_lane;
    for (;;) {
      const size_t i = next.fetch_add(1);
      if (i >= next_end) break;
      size_t olen = 0;
      uint32_t crc = 0;
      const int rc = deflate_member_on((const uint8_t *)g.d_in.p + din[i], (size_t)in_len[i], level, window_bits,
                                       (uint8_t *)g.d_out.p + dout[i], dout[i + 1] - dout[i], ws, ws_lane, s, &olen, &crc,
                                       pre.empty() || in_len[i] == 0 ? nullptr : &pre[i]);
      if (rc) return fail(rc);
      out_len[i] = olen;
      if (crc32) crc32[i] = crc;
      if (olen > out_cap[i]) {
        status[i] = B200Z_U_NOSPC;
        continue;
      }
      status[i] = B200Z_OK;
      if (olen && cudaMemcpyAsync(out_base + out_off[i], (uint8_t *)g.d_out.p + dout[i], olen, cudaMemcpyDeviceToHost, s) !=
                      cudaSuccess)
        return fail(B200Z_E_NODEVICE);
    }
    if (cudaStreamSynchronize(s) != cudaSuccess) fail(B200Z_E_NODEVICE);
  };
  auto run_lanes = [&]() {
    if (lanes == 1) {
      lane(0);
    } else {
      std::vector<std::thread> th;
      for (size_t l = 1; l < lanes; ++l) th.emplace_back(lane, l);
      lane(0);
      for (auto &t : th) t.join();
    }
  };
  if (level >= 1 && level <= 3) {
    // _deflateFast is one serial chain per member; the batch is the parallel axis: ONE launch makes the tokens of a whole
    // group of members (a warp per member, deflate_kernels.cu: k_defl_fast_batch), then the lanes cut the blocks, build
    // the trees and emit the bits of each.  A group is as many members as the token store holds (12 bytes per input
    // byte; B200Z_DEFLATE_TOK_MB, default 49152).
    size_t budget = (size_t)48 << 30;
    {
      size_t free_b = 0, total_b = 0;  // (never more than 60 % of what the device has free right now)
      if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && free_b) budget = std::min(budget, free_b / 10 * 6 + g.d_tok.cap);
    }
    if (const char *e = getenv("B200Z_DEFLATE_TOK_MB")) budget = std::max<size_t>(1, (size_t)atoll(e)) << 20;
    pre.assign(n_units, DeflFastMember());
    size_t lo = 0;
    auto failed = [&]() {
      for (size_t l = 0; l < lanes; ++l)
        if (lane_rc[l]) return true;
      return false;
    };
    while (lo < n_units && !failed()) {
      size_t hi = lo, bytes = 256;
      std::vector<size_t> off;
      while (hi < n_units) {
        const size_t need = align_up(((size_t)in_len[hi] + 2) * 4, 256) * 3 + 256;
        if (hi > lo && bytes + need > budget) break;
        off.push_back(bytes);
        bytes += need;
        hi++;
      }
      const size_t list_off = align_up(bytes, 256);
      bytes = list_off + (hi - lo) * sizeof(DeflFastMember);
      CU(g.d_tok.reserve(bytes));
      std::vector<DeflFastMember> order;
      for (size_t i = lo; i < hi; ++i) {
        const size_t n = (size_t)in_len[i], a = align_up((n + 2) * 4, 256);
        uint8_t *base = (uint8_t *)g.d_tok.p + off[i - lo];
        DeflFastMember m;
        m.d = (const uint8_t *)g.d_in.p + din[i];
        m.n = (uint32_t)n;
        m.tok = (uint32_t *)base;
        m.tally_ss = (uint32_t *)(base + a);
        m.next_ss = (uint32_t *)(base + 2 * a);
        m.ntok = (uint32_t *)(base + 3 * a);
        pre[i] = m;
        if (n) order.push_back(m);
      }
      std::stable_sort(order.begin(), order.end(), [](const DeflFastMember &x, const DeflFastMember &y) { return x.n > y.n; });
      if (!order.empty()) {
        CU(cudaStreamWaitEvent(g.stream, staged, 0));
        CU(cudaMemcpyAsync((uint8_t *)g.d_tok.p + list_off, order.data(), order.size() * sizeof(DeflFastMember),
                           cudaMemcpyHostToDevice, g.stream));
        CU(deflate_fast_tokens_batch((const DeflFastMember *)((uint8_t *)g.d_tok.p + list_off), (uint32_t)order.size(), level,
                                     window_bits, (uint32_t *)g.d_tok.p, g.stream));
        CU(cudaStreamSynchronize(g.stream));
      }
      next.store(lo);
      next_end = hi;
      run_lanes();
      lo = hi;
    }
  } else {
    run_lanes();
  }
  cudaEventDestroy(staged);
  for (size_t l = 0; l < lanes; ++l)
    if (lane_rc[l]) {
      set_err("deflate_batch: %s", lane_err[l].empty() ? "a lane failed" : lane_err[l].c_str());
      return lane_rc[l];
    }
  return B200Z_OK;
}

}  // namespace b200z

using namespace b200z;

// =============================================================================================
// C ABI
// =============================================================================================

// ---------------------------------------------------------------------------------------------
// ZIP container (SURVEY.md 8f2): directory parse on the host, members as ONE inflate batch
// ---------------------------------------------------------------------------------------------
static inline uint64_t le64(const uint8_t *p) { return (uint64_t)le32(p) | ((uint64_t)le32(p + 4) << 32); }

// ZipDirectory._findSignature (zip_directory.dart:139-182): 1024-byte chunks from the end, each scanned backwards; a
// signature that straddles two chunks, or lies in the last 4 bytes, is not seen.
static long long zip_find_eocd(const uint8_t *z, size_t len) {
  if (len <= 4) return -1;
  const long long length = (long long)len - 4;
  const long long chunk = length < 1024 ? length : 1024;
  long long start = length - chunk;
  while (start >= 0) {
    for (long long cp = chunk - 4; cp >= 0; --cp)
      if (le32(z + start + cp) == 0x06054b50u) return start + cp;
    if (start > 0 && start < chunk) start = 0;
    else start -= chunk;
  }
  return -1;
}

extern "C" int b200z_zip_list(const uint8_t *z, size_t len, b200z_zip_entry *entries, size_t cap, size_t *n_entries) {
  if (n_entries) *n_entries = 0;
  if (!z && len) return B200Z_E_ARG;
  const long long fp = zip_find_eocd(z, len);
  if (fp < 0) return B200Z_OK;  // ZipDirectory.read returns with no headers (zip_directory.dart:26-29)
  // (overflow-safe: positions and sizes come from the archive as full 64-bit values)
#define ZNEED_IN(pos, k, lim)                                                       \
  if ((unsigned long long)(pos) > (unsigned long long)(lim) ||                      \
      (unsigned long long)(k) > (unsigned long long)(lim) - (unsigned long long)(pos)) { \
    set_err("zip: read past the end at %llu (Dart: RangeError)", (unsigned long long)(pos)); \
    return B200Z_E_THROW;                                                          \
  }
#define ZNEED(pos, k) ZNEED_IN(pos, k, len)
  ZNEED(fp, 22);
  uint64_t cd_size = le32(z + fp + 12), cd_off = le32(z + fp + 16);
  {
    const size_t clen = le16(z + fp + 20);
    ZNEED(fp + 22, clen);  // the comment is read (readString) before the zip64 records are looked at
  }
  // _readZip64Data :65-137
  if (fp >= 20 && le32(z + fp - 20) == 0x07064b50u) {
    const uint64_t z64 = le64(z + fp - 20 + 8);
    if (z64 <= len && len - z64 >= 4 && le32(z + z64) == 0x06064b50u) {
      ZNEED(z64, 56);
      cd_size = le64(z + z64 + 40);
      cd_off = le64(z + z64 + 48);
    } else if (z64 > len || len - z64 < 4) {
      ZNEED(z64, 4);
    }
  }
  // central directory :50-63
  size_t n = 0;
  uint64_t p = cd_off;
  // dirContent = input.subset(position: offset, length: size) (input_memory_stream.dart:15-27,111-119): a length that
  // reaches beyond the archive is cut to what is there; an offset beyond it, or a negative (>= 2^63) offset or size, makes
  // Uint8List.view throw.  The headers are then read from that sub-stream: running over ITS end throws.
  if (cd_off > len || (cd_size >> 63) != 0) {
    set_err("zip: central directory at %llu (+%llu) lies outside the archive (Dart: RangeError)", (unsigned long long)cd_off,
            (unsigned long long)cd_size);
    return B200Z_E_THROW;
  }
  const uint64_t cd_end = cd_size > len - cd_off ? (uint64_t)len : cd_off + cd_size;
#define DNEED(pos, k) ZNEED_IN(pos, k, cd_end)
  while (p < cd_end) {
    DNEED(p, 4);
    if (le32(z + p) != 0x02014b50u) break;
    DNEED(p, 46);
    // ZipFileHeader.read (zip_file_header.dart:28-111)
    const uint8_t *h = z + p;
    b200z_zip_entry e;
    memset(&e, 0, sizeof e);
    e.version_made_by = le16(h + 4);
    uint64_t comp = le32(h + 20), uncomp = le32(h + 24), lho = le32(h + 42);
    const size_t fn_len = le16(h + 28), ex_len = le16(h + 30), cm_len = le16(h + 32);
    uint32_t disk = le16(h + 34);
    e.ext_attr = le32(h + 38);
    DNEED(p + 46, fn_len + ex_len + cm_len);
    e.cd_name_off = p + 46;
    e.cd_name_len = (uint32_t)fn_len;
    if (ex_len >= 4) {  // :48-98 -- shorter extra fields are ignored
      const uint8_t *x = h + 46 + fn_len;
      size_t xo = 0;
      while (ex_len - xo >= 4) {
        const uint32_t id = le16(x + xo);
        size_t size = le16(x + xo + 2);
        xo += 4;
        if (xo + size > ex_len) {
          set_err("zip: extra field overruns its record (Dart: RangeError)");
          return B200Z_E_THROW;
        }
        if (id == 1) {
          size_t q = xo;
          if (size >= 8 && uncomp == 0xffffffffu) { uncomp = le64(x + q); q += 8; size -= 8; }
          if (size >= 8 && comp == 0xffffffffu) { comp = le64(x + q); q += 8; size -= 8; }
          if (size >= 8 && lho == 0xffffffffu) { lho = le64(x + q); q += 8; size -= 8; }
          if (size >= 4 && disk == 0xffffu) { disk = le32(x + q); q += 4; size -= 4; }
          xo = q + size;
        } else {
          xo += size;
        }
      }
    }
    (void)disk;
    p += 46 + fn_len + ex_len + cm_len;
    // ZipFile.read at the local header (zip_file.dart:73-149)
    e.local_header_off = lho;
    e.comp_size = comp;
    e.uncomp_size = uncomp;
    e.hint_uncomp_size = uncomp;
    ZNEED(lho, 4);
    if (le32(z + lho) == 0x04034b50u) {
      ZNEED(lho, 30);
      const uint8_t *l = z + lho;
      e.flags = le16(l + 6);
      e.method = le16(l + 8);
      e.mod_time = le16(l + 10);
      e.mod_date = le16(l + 12);
      e.crc32 = le32(l + 14);
      const size_t lfn = le16(l + 26), lex = le16(l + 28);
      ZNEED(lho + 30, lfn + lex);
      e.name_off = lho + 30;
      e.name_len = (uint32_t)lfn;
      e.data_off = lho + 30 + lfn + lex;
      e.has_data = 1;
      if ((comp >> 63) != 0) {  // readBytes(negative count): Uint8List.view throws
        set_err("zip: compressed size %llu (Dart: RangeError)", (unsigned long long)comp);
        return B200Z_E_THROW;
      }
      if (comp > len - e.data_off) {  // readBytes hands out what is there (data_off <= len: checked above)
        e.comp_size = len - e.data_off;
      }
      if (e.flags & 0x08) {  // data descriptor :137-148: CRC and the 32-bit sizes are replaced by what follows the data
        uint64_t q = e.data_off + e.comp_size;
        ZNEED(q, 4);
        const uint32_t sig_or_crc = le32(z + q);
        q += 4;
        if (sig_or_crc == 0x08074b50u) {
          ZNEED(q, 4);
          e.crc32 = le32(z + q);
          q += 4;
        } else {
          e.crc32 = sig_or_crc;
        }
        ZNEED(q, 8);
        e.uncomp_size = le32(z + q + 4);
      }
    }
    if (n < cap && entries) entries[n] = e;
    n++;
  }
#undef DNEED
#undef ZNEED
#undef ZNEED_IN
  if (n_entries) *n_entries = n;
  if (n > cap && entries) {
    set_err("zip: %zu entries, capacity %zu", n, cap);
    return B200Z_E_NOSPC;
  }
  return B200Z_OK;
}

// ZipDirectory.zipFileComment (zip_directory.dart:41-44): byte range of the archive comment, or length 0
extern "C" int b200z_zip_comment(const uint8_t *z, size_t len, uint64_t *off, uint32_t *clen) {
  if (off) *off = 0;
  if (clen) *clen = 0;
  const long long fp = zip_find_eocd(z, len);
  if (fp < 0) return B200Z_OK;
  if ((unsigned long long)fp + 22 > len) {
    set_err("zip: read past the end at %lld (Dart: RangeError)", fp);
    return B200Z_E_THROW;
  }
  const uint32_t n = le16(z + fp + 20);
  if ((unsigned long long)fp + 22 + n > len) {
    set_err("zip: comment overruns the archive (Dart: RangeError)");
    return B200Z_E_THROW;
  }
  if (off) *off = (uint64_t)fp + 22;
  if (clen) *clen = n;
  return B200Z_OK;
}

extern "C" int b200z_zip_extract(const uint8_t *z, size_t len, const b200z_zip_entry *entries, size_t n, uint8_t *out,
                                 size_t out_cap, const uint64_t *out_off, const uint64_t *out_room, uint64_t *out_len,
                                 int32_t *status, uint32_t flags) {
  int rc = require_init();
  if (rc) return rc;
  if (n == 0) return B200Z_OK;
  if (!entries || !out_off || !out_room || !out_len || !status) return B200Z_E_ARG;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  // members: deflate -> one inflate batch; stored (and unknown methods, which the reference treats as stored,
  // zip_file.dart:83) -> device copies; bzip2 -> one stream each, afterwards
  std::vector<uint64_t> u_in_off, u_out_off;
  std::vector<uint32_t> u_in_len, u_cap, u_idx;
  std::vector<size_t> bz_idx;
  uint64_t lo = ~0ull, hi = 0;
  for (size_t i = 0; i < n; ++i) {
    const b200z_zip_entry &e = entries[i];
    out_len[i] = 0;
    status[i] = B200Z_U_DONE;
    if (!e.has_data) continue;
    if (e.flags & 1u) {
      status[i] = B200Z_ZIP_ENCRYPTED;
      continue;
    }
    if (out_off[i] > out_cap || out_room[i] > out_cap - out_off[i] || e.data_off > len || e.comp_size > len - e.data_off) {
      set_err("zip_extract: entry %zu lies outside the buffers", i);
      return B200Z_E_ARG;
    }
    if (e.method == 8 || e.method == 12) {
      if (e.comp_size > 0xfffffff0ull || out_room[i] > 0xfffffff0ull) {
        status[i] = B200Z_ZIP_TOO_LARGE;
        continue;
      }
    }
    if (e.method == 12) {
      bz_idx.push_back(i);
      continue;
    }
    if (out_room[i]) {
      lo = out_off[i] < lo ? out_off[i] : lo;
      hi = out_off[i] + out_room[i] > hi ? out_off[i] + out_room[i] : hi;
    }
    if (e.method == 8) {
      // ZipFile.getStream: ZLibDecoder().decodeBytes(compressed, raw: true) on exactly the member's bytes.  On the Dart
      // VM that is dart:io's zlib; the pure-Dart Inflate wants maxCodeLength bits after the last code (SURVEY Q1) and
      // so can drop the last symbols of such a stream.  Default: what the VM gives -- a few bytes that follow the
      // member are made readable so the lookahead is satisfied; B200Z_ZIP_WEB_EOS: the pure-Dart behaviour.
      uint64_t pad = 0;
      if (!(flags & B200Z_ZIP_WEB_EOS)) {
        pad = len - (e.data_off + e.comp_size);
        if (pad > 8) pad = 8;
      }
      u_in_off.push_back(e.data_off);
      u_in_len.push_back((uint32_t)(e.comp_size + pad));
      u_out_off.push_back(out_off[i]);
      u_cap.push_back((uint32_t)out_room[i]);
      u_idx.push_back((uint32_t)i);
    }
  }
  const bool any_dev = hi > lo;
  if (any_dev || !u_idx.empty()) {
    rc = stage_input(z, len);
    if (rc) return rc;
    CU(cudaMemsetAsync((uint8_t *)g.d_in.p + len, 0, 64, g.stream));
    CU(g.d_out.reserve((hi ? hi : 1) + 64));
  }
  for (size_t i = 0; i < n; ++i) {
    const b200z_zip_entry &e = entries[i];
    if (!e.has_data || (e.flags & 1u) || e.method == 8 || e.method == 12) continue;
    uint64_t k = e.comp_size < out_room[i] ? e.comp_size : out_room[i];
    if (k) CU(cudaMemcpyAsync((uint8_t *)g.d_out.p + out_off[i], (const uint8_t *)g.d_in.p + e.data_off, k, cudaMemcpyDeviceToDevice, g.stream));
    out_len[i] = e.comp_size;
    if (e.comp_size > out_room[i]) status[i] = B200Z_U_NOSPC;
  }
  // ---- flush points: a member that was written with Z_FULL_FLUSH every so often is many independent raw DEFLATE
  // streams back to back (each ends with the byte-aligned empty stored block 00 00 FF FF and restarts the window).
  // Candidates are found by a byte scan and PROVEN by a sizing pass (count-only decode of every piece: a piece must end
  // exactly on its marker at a block boundary and must not reach back before its own start -- which also rejects
  // Z_SYNC_FLUSH points, whose window continues); a member with any doubtful piece is decoded whole.
  if (!u_idx.empty() && !(flags & B200Z_ZIP_NO_SPLIT)) {
    bool worth = false;
    for (size_t k = 0; k < u_idx.size(); ++k) worth = worth || u_in_len[k] >= (256u << 10);
    if (worth) {
      const uint32_t ccap = 1u << 22;
      CU(g.d_small.reserve((size_t)ccap * 8 + 256));
      unsigned long long *d_list = (unsigned long long *)((uint8_t *)g.d_small.p + 256);
      uint32_t *d_cnt = (uint32_t *)g.d_small.p;
      CU(launch_find_markers((const uint8_t *)g.d_in.p, len, d_list, d_cnt, ccap, g.stream));
      uint32_t ncand = 0;
      CU(cudaMemcpyAsync(&ncand, d_cnt, 4, cudaMemcpyDeviceToHost, g.stream));
      CU(cudaStreamSynchronize(g.stream));
      if (ncand > 0 && ncand <= ccap) {
        std::vector<unsigned long long> cand(ncand);
        CU(cudaMemcpy(cand.data(), d_list, (size_t)ncand * 8, cudaMemcpyDeviceToHost));
        std::sort(cand.begin(), cand.end());
        // pieces of every big member
        std::vector<uint64_t> s_in_off, s_out_off;
        std::vector<uint32_t> s_in_len, s_cap, s_member, first_seg(u_idx.size() + 1, 0);
        for (size_t k = 0; k < u_idx.size(); ++k) {
          first_seg[k] = (uint32_t)s_in_off.size();
          if (u_in_len[k] < (256u << 10)) continue;
          const uint64_t a0 = u_in_off[k], a1 = a0 + entries[u_idx[k]].comp_size, aend = a0 + u_in_len[k];
          auto it = std::upper_bound(cand.begin(), cand.end(), a0);
          uint64_t start = a0;
          size_t pieces = 0;
          for (; it != cand.end() && *it < a1; ++it) {
            if (*it - start < 4096) continue;  // not worth a unit of its own
            s_in_off.push_back(start);
            s_in_len.push_back((uint32_t)(*it - start));
            s_member.push_back((uint32_t)k);
            start = *it;
            pieces++;
          }
          if (pieces == 0) continue;
          s_in_off.push_back(start);
          s_in_len.push_back((uint32_t)(aend - start));
          s_member.push_back((uint32_t)k);
        }
        first_seg[u_idx.size()] = (uint32_t)s_in_off.size();
        const size_t ns = s_in_off.size();
        if (ns) {
          s_out_off.assign(ns, 0);
          s_cap.assign(ns, 0xfffffff0u);
          std::vector<uint32_t> a_len(ns), a_used(ns);
          std::vector<int32_t> a_st(ns);
          rc = run_batch_on_staged(s_in_off.data(), s_in_len.data(), s_out_off.data(), s_cap.data(), a_len.data(), a_st.data(),
                                   a_used.data(), ns, 0, true);
          if (rc) return rc;
          // rebuild the unit list: proven members contribute their pieces, the others stay whole
          std::vector<uint64_t> n_in_off, n_out_off;
          std::vector<uint32_t> n_in_len, n_cap, n_idx;
          for (size_t k = 0; k < u_idx.size(); ++k) {
            const uint32_t f = first_seg[k], l = first_seg[k + 1];
            bool ok = l > f;
            uint64_t total = 0;
            for (uint32_t q = f; q < l && ok; ++q) {
              const bool last = q + 1 == l;
              ok = last ? (a_st[q] == B200Z_U_DONE) : (a_st[q] == B200Z_U_EOS && a_used[q] == s_in_len[q]);
              total += a_len[q];
            }
            ok = ok && total <= u_cap[k];
            if (!ok) {
              n_in_off.push_back(u_in_off[k]); n_in_len.push_back(u_in_len[k]); n_out_off.push_back(u_out_off[k]);
              n_cap.push_back(u_cap[k]); n_idx.push_back(u_idx[k]);
              continue;
            }
            uint64_t o = u_out_off[k];
            for (uint32_t q = f; q < l; ++q) {
              n_in_off.push_back(s_in_off[q]); n_in_len.push_back(s_in_len[q]); n_out_off.push_back(o);
              n_cap.push_back(a_len[q]); n_idx.push_back(u_idx[k] | (q + 1 == l ? 0u : 0x80000000u));
              o += a_len[q];
            }
          }
          u_in_off.swap(n_in_off); u_in_len.swap(n_in_len); u_out_off.swap(n_out_off); u_cap.swap(n_cap); u_idx.swap(n_idx);
        }
      }
    }
  }
  size_t early_to = (size_t)lo;  // output bytes [lo, early_to) are on their way to the host already (copy stream)
  if (!u_idx.empty()) {
    const size_t m = u_idx.size();
    std::vector<uint32_t> r_len(m), r_used(m);
    std::vector<int32_t> r_st(m);
    // A large archive is decoded in chunks of units (in output order), and the bytes of a finished chunk -- with the stored
    // members that lie between its units -- go to the host on the copy stream while the next chunk is decoded
    // (B200Z_ZIP_CHUNKS, default 8 from 512 MiB of output on; 1: one batch, one copy at the end).
    size_t nchunks = (hi - lo) >= ((size_t)512 << 20) ? 8 : 1;
    if (const char *ce = getenv("B200Z_ZIP_CHUNKS")) nchunks = (size_t)std::max(1, atoi(ce));
    for (size_t k = 1; k < m && nchunks > 1; ++k)
      if (u_out_off[k] < u_out_off[k - 1]) nchunks = 1;  // (units are made in output order; if ever not, no early copies)
    if (nchunks > m) nchunks = m;
    for (size_t c = 0, k0 = 0; c < nchunks; ++c) {
      const size_t k1 = m * (c + 1) / nchunks;
      if (k1 == k0) continue;
      rc = run_batch_on_staged(u_in_off.data() + k0, u_in_len.data() + k0, u_out_off.data() + k0, u_cap.data() + k0, r_len.data() + k0,
                               r_st.data() + k0, r_used.data() + k0, k1 - k0, (size_t)hi);
      if (rc) {
        if (early_to > lo) cudaStreamSynchronize(g.s_d2h);
        return rc;
      }
      const size_t end = k1 < m ? (size_t)u_out_off[k1] : (size_t)hi;
      if (nchunks > 1 && end > early_to && end <= hi) {
        CU(cudaMemcpyAsync(out + early_to, (const uint8_t *)g.d_out.p + early_to, end - early_to, cudaMemcpyDeviceToHost, g.s_d2h));
        early_to = end;
      }
      k0 = k1;
    }
    for (size_t k = 0; k < m; ++k) {
      const uint32_t i = u_idx[k] & 0x7fffffffu;
      const bool inner = (u_idx[k] & 0x80000000u) != 0;  // a piece that is not the member's last
      out_len[i] += r_len[k];
      if (!inner) {
        if (status[i] == B200Z_U_DONE) status[i] = r_st[k];
      } else if (!(r_st[k] == B200Z_U_EOS && r_len[k] == u_cap[k])) {
        status[i] = r_st[k] == B200Z_U_EOS || r_st[k] == B200Z_U_DONE ? B200Z_U_STOP : r_st[k];  // cannot happen after the sizing pass
      }
    }
  }
  if (any_dev) {
    if (hi > early_to)
      CU(cudaMemcpyAsync(out + early_to, (const uint8_t *)g.d_out.p + early_to, hi - early_to, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    if (early_to > lo) CU(cudaStreamSynchronize(g.s_d2h));
  }
  for (size_t i : bz_idx) {  // BZip2Decoder().decodeStream(_rawContent, output) (zip_file.dart:189-192,239-245)
    const b200z_zip_entry &e = entries[i];
    size_t got = 0;
    rc = bzip2_decode_impl(z + e.data_off, (size_t)e.comp_size, 0, out + out_off[i], (size_t)out_room[i], &got);
    out_len[i] = got;
    status[i] = rc == B200Z_OK ? B200Z_U_DONE : rc == B200Z_E_NOSPC ? B200Z_U_NOSPC : rc == B200Z_E_THROW ? B200Z_U_THROW : B200Z_U_STOP;
  }
  return B200Z_OK;
}

extern "C" {

const char *b200z_version(void) { return "b200z 0.1 (sm_100a)"; }
const char *b200z_last_error(void) { return t_err; }
uint64_t b200z_launch_count(void) { return g_launches.load(); }
// (debug, not part of the ABI) BZip2 candidate blocks decoded by k_bz2_entropy_fast / left to the exact kernel so far
void b200z_debug_bz2_blocks(unsigned long long out[2]) {
  out[0] = g_bz2_fast_blocks.load();
  out[1] = g_bz2_exact_blocks.load();
}

int b200z_bzip2_decode(const uint8_t *in, size_t in_len, int verify, uint8_t *out, size_t out_cap, size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  size_t n = 0;
  rc = bzip2_decode_impl(in, in_len, verify, out, out_cap, &n);
  if (out_len) *out_len = n;
  return rc;
}
void b200z_profile_enable(int on) { profile_enable(on != 0); }
int b200z_crc32(const uint8_t *in, size_t in_len, uint32_t *crc) {
  int rc = require_init();
  if (rc) return rc;
  if (!crc) return B200Z_E_ARG;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  rc = stage_input(in, in_len);
  if (rc) return rc;
  return device_crc32((const uint8_t *)g.d_in.p, in_len, crc);
}

int b200z_bzip2_decode_shard(const uint8_t *in, size_t in_len, uint32_t rank, uint32_t world, uint8_t *out, size_t out_cap,
                             size_t *out_len, b200z_bz2_block *blocks, size_t blocks_cap, size_t *n_blocks) {
  int rc = require_init();
  if (rc) return rc;
  if (world == 0 || rank >= world || !blocks) {
    set_err("bzip2_decode_shard: bad rank/world");
    return B200Z_E_ARG;
  }
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  Bz2Shard sh{rank, world, blocks, blocks_cap, 0};
  size_t n = 0;
  rc = bzip2_decode_impl(in, in_len, 0, out, out_cap, &n, &sh);
  if (out_len) *out_len = n;
  if (n_blocks) *n_blocks = sh.n_blocks;
  return rc;
}

int b200z_bzip2_encode(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap, size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  if (in_len >= 0xfff00000ull) {
    set_err("bzip2 encode: inputs of 4 GiB and more are not supported");
    return B200Z_E_ARG;
  }
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  rc = stage_input(in, in_len);
  if (rc) return rc;
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  const size_t budget = free_b + g.d_ws.cap > ((size_t)2 << 30) ? (free_b + g.d_ws.cap) / 2 : ((size_t)1 << 30);
  const bz2e::Plan plan = bz2e::plan(in_len, budget < ((size_t)24 << 30) ? budget : ((size_t)24 << 30));
  const size_t cap = align_up(bz2e::bound(in_len) + 64, 256);
  CU(g.d_out.reserve(cap));
  CU(g.d_ws.reserve(plan.ws_bytes));
  size_t n = 0;
  bz2e::Stats st;
  int r = bz2e::encode_device((const uint8_t *)g.d_in.p, in_len, (uint8_t *)g.d_out.p, cap, g.d_ws.p, plan, &n, &st,
                              (void *)g.stream);
  if (r == -3) {
    set_err("bzip2 encode: internal output bound too small (%zu)", cap);
    return B200Z_E_INTERNAL;
  }
  if (r != 0) {
    cudaError_t e = cudaGetLastError();
    set_err("bzip2 encode: device failure (%s)", cudaGetErrorString(e));
    return B200Z_E_INTERNAL;
  }
  if (out_len) *out_len = n;
  if (n > out_cap) {
    set_err("bzip2 encode: output needs %zu bytes, out_cap %zu", n, out_cap);
    return B200Z_E_NOSPC;
  }
  CU(cudaMemcpyAsync(out, g.d_out.p, n, cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  return B200Z_OK;
}
size_t b200z_bzip2_bound(size_t in_len) { return bz2e::bound(in_len); }

int b200z_profile_read(double *fast_ms, double *decode_ms, double *expand_ms, uint64_t *n_batches) {
  return profile_read(fast_ms, decode_ms, expand_ms, n_batches) ? B200Z_E_NODEVICE : B200Z_OK;
}

int b200z_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int b200z_init(int device, uint32_t flags) {
  (void)flags;
  std::lock_guard<std::mutex> lk(g.mu);
  if (g.inited && g.device == device) return B200Z_OK;
  int n = b200z_device_count();
  if (n <= 0 || device < 0 || device >= n) {
    set_err("b200z_init: CUDA device %d not available (%d visible): there is no CPU fallback", device, n);
    return B200Z_E_NODEVICE;
  }
  CU(cudaSetDevice(device));
  if (!g.stream) {
    CU(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&g.s_h2d, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&g.s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < Ctx::kCompStreams; ++i) CU(cudaStreamCreateWithFlags(&g.s_comp[i], cudaStreamNonBlocking));
  }
  g.device = device;
  g.inited = true;
  return B200Z_OK;
}

void b200z_shutdown(void) {
  file_release();  // before g.mu: a file call holds its own lock while it takes g.mu, never the other way round
  std::lock_guard<std::mutex> lk(g.mu);
  if (!g.inited) return;
  cudaSetDevice(g.device);
  cudaStreamSynchronize(g.stream);
  g.d_in.release(); g.d_out.release(); g.d_ws.release(); g.d_meta.release(); g.d_small.release(); g.d_bz.release(); g.d_tok.release();
  g.h_meta.release();
  cudaStreamDestroy(g.stream);
  cudaStreamDestroy(g.s_h2d);
  cudaStreamDestroy(g.s_d2h);
  for (int i = 0; i < Ctx::kCompStreams; ++i) cudaStreamDestroy(g.s_comp[i]);
  g.stream = g.s_h2d = g.s_d2h = nullptr;
  g.inited = false;
}

void *b200z_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    set_err("b200z_host_alloc(%zu) failed", bytes);
    return nullptr;
  }
  return p;
}
void b200z_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

size_t b200z_inflate_workspace_bytes(size_t n_units, size_t total_in_bytes, size_t out_extent) {
  (void)total_in_bytes;
  return workspace_bytes(n_units, out_extent);
}

int b200z_inflate_batch_device(const uint8_t *d_in_base, const uint64_t *d_in_off, const uint32_t *d_in_len,
                               uint8_t *d_out_base, const uint64_t *d_out_off, const uint32_t *d_out_cap,
                               uint32_t *d_out_len, int32_t *d_status, uint32_t *d_in_used, size_t n_units,
                               void *d_workspace, size_t workspace_bytes_, void *cuda_stream) {
  int rc = require_init();
  if (rc) return rc;
  if (n_units == 0) return B200Z_OK;
  const size_t extent = inflate_ws_extent_for(n_units, workspace_bytes_);
  if (extent == 0) {
    set_err("inflate_batch_device: workspace too small (size it with b200z_inflate_workspace_bytes)");
    return B200Z_E_ARG;
  }
  InflateBatch b;
  b.in_base = d_in_base; b.in_off = d_in_off; b.in_len = d_in_len;
  b.out_base = d_out_base; b.out_off = d_out_off; b.out_cap = d_out_cap;
  b.out_len = d_out_len; b.status = d_status; b.in_used = d_in_used;
  b.n_units = n_units;
  b.ws = inflate_ws_carve(d_workspace, n_units, extent);
  cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : g.stream;
  CU(launch_inflate(b, s));
  return B200Z_OK;
}

int b200z_inflate_batch(const uint8_t *in_base, size_t in_bytes, const uint64_t *in_off, const uint32_t *in_len,
                        uint8_t *out_base, size_t out_bytes, const uint64_t *out_off, const uint32_t *out_cap,
                        uint32_t *out_len, int32_t *status, uint32_t *in_used, size_t n_units) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  for (size_t u = 0; u < n_units; ++u) {
    if (in_off[u] + in_len[u] > in_bytes || out_off[u] + out_cap[u] > out_bytes) {
      set_err("inflate_batch: unit %zu exceeds the buffers", u);
      return B200Z_E_ARG;
    }
  }
  rc = stage_input(in_base, in_bytes);
  if (rc) return rc;
  CU(g.d_out.reserve(out_bytes + 64));
  rc = run_batch_on_staged(in_off, in_len, out_off, out_cap, out_len, status, in_used, n_units, out_bytes);
  if (rc) return rc;
  // only the units' slots: the bytes between them are the caller's (the device buffer there holds earlier calls' data)
  CU(copy_slots_to_host(out_base, (const uint8_t *)g.d_out.p, 0, out_off, out_cap, n_units, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  return B200Z_OK;
}

int b200z_inflate_raw(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap, size_t *out_len,
                      size_t *in_consumed, int32_t *unit_status) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  if (in_len > 0xfffffff0u) {
    set_err("inflate_raw: streams above 4 GiB are not supported");
    return B200Z_E_ARG;
  }
  rc = stage_input(in, in_len);
  if (rc) return rc;
  OneResult r{0, 0, B200Z_U_EOS};
  if (in_len > 0) {
    rc = run_one_staged(0, in_len, 0, out_cap, &r);
    if (rc) return rc;
    if (r.out_len) CU(cudaMemcpyAsync(out, g.d_out.p, r.out_len, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
  }
  if (out_len) *out_len = r.out_len;
  if (in_consumed) *in_consumed = r.in_used;
  if (unit_status) *unit_status = r.status;
  if (r.status == B200Z_U_NOSPC) {
    set_err("inflate_raw: out_cap %zu too small", out_cap);
    return B200Z_E_NOSPC;
  }
  if (r.status == B200Z_U_RANGE || r.status == B200Z_U_THROW) {
    set_err("inflate_raw: Dart would throw RangeError (unit status %d)", r.status);
    return B200Z_E_THROW;
  }
  return B200Z_OK;  // STOP / BADCODE: reference keeps the partial output silently
}

int b200z_deflate_raw(const uint8_t *in, size_t in_len, int level, int window_bits, uint8_t *out, size_t out_cap,
                      size_t *out_len, uint32_t *crc32_of_input) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  rc = stage_input(in, in_len);
  if (rc) return rc;
  CU(cudaMemsetAsync((uint8_t *)g.d_in.p + in_len, 0, 64, g.stream));
  size_t n = 0;
  rc = deflate_staged(in_len, level, window_bits, &n);
  if (rc) return rc;
  if (out_len) *out_len = n;
  if (n > out_cap) {
    set_err("deflate: output needs %zu bytes, out_cap %zu", n, out_cap);
    return B200Z_E_NOSPC;
  }
  if (n) CU(cudaMemcpyAsync(out, g.d_out.p, n, cudaMemcpyDeviceToHost, g.stream));
  if (crc32_of_input) {
    rc = device_crc32((const uint8_t *)g.d_in.p, in_len, crc32_of_input);
    if (rc) return rc;
  }
  CU(cudaStreamSynchronize(g.stream));
  return B200Z_OK;
}

size_t b200z_deflate_bound(size_t in_len) { return deflate_bound(in_len) + 32; }

int b200z_deflate_batch(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len, size_t n_units, int level,
                        int window_bits, uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap, uint64_t *out_len,
                        uint32_t *crc32, int32_t *status) {
  int rc = require_init();
  if (rc) return rc;
  if (window_bits < 9 || window_bits > 15 || level < 0 || level > 9) {
    set_err("deflate: invalid level %d / windowBits %d (Dart: LateInitializationError)", level, window_bits);
    return B200Z_E_ARG;
  }
  if (n_units == 0) return B200Z_OK;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  return deflate_batch_impl(in_base, in_off, in_len, n_units, level, window_bits, out_base, out_off, out_cap, out_len, crc32,
                            status);
}

int b200z_zlib_encode(const uint8_t *in, size_t in_len, int level, int window_bits, int raw, uint8_t *out, size_t out_cap,
                      size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  rc = stage_input(in, in_len);
  if (rc) return rc;
  CU(cudaMemsetAsync((uint8_t *)g.d_in.p + in_len, 0, 64, g.stream));
  size_t n = 0;
  rc = deflate_staged(in_len, level, window_bits, &n);
  if (rc) return rc;
  const size_t total = raw ? n : n + 6;
  if (out_len) *out_len = total;
  if (total > out_cap) {
    set_err("zlib_encode: output needs %zu bytes, out_cap %zu", total, out_cap);
    return B200Z_E_NOSPC;
  }
  size_t o = 0;
  if (!raw) {
    // CMF / FLG with FLEVEL 0 for every level (_zlib_encoder_web.dart:44-60, quirk Q4)
    int wb = window_bits < 0 ? 0 : window_bits > 15 ? 15 : window_bits;
    int cmf = ((wb - 8) << 4) | 8, flag = 0, fcheck = 0;
    while ((cmf * 256 + (flag | fcheck)) % 31 != 0) fcheck++;
    out[o++] = (uint8_t)cmf;
    out[o++] = (uint8_t)(flag | fcheck);
  }
  if (n) CU(cudaMemcpyAsync(out + o, g.d_out.p, n, cudaMemcpyDeviceToHost, g.stream));
  o += n;
  if (!raw) {
    uint32_t ad;
    rc = device_adler32((const uint8_t *)g.d_in.p, in_len, &ad);
    if (rc) return rc;
    out[o++] = (uint8_t)(ad >> 24);
    out[o++] = (uint8_t)(ad >> 16);
    out[o++] = (uint8_t)(ad >> 8);
    out[o++] = (uint8_t)ad;
  }
  CU(cudaStreamSynchronize(g.stream));
  return B200Z_OK;
}

int b200z_gzip_encode(const uint8_t *in, size_t in_len, int level, uint32_t mtime, uint8_t *out, size_t out_cap,
                      size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  rc = stage_input(in, in_len);
  if (rc) return rc;
  CU(cudaMemsetAsync((uint8_t *)g.d_in.p + in_len, 0, 64, g.stream));
  size_t n = 0;
  rc = deflate_staged(in_len, level, 15, &n);
  if (rc) return rc;
  const size_t total = n + 18;
  if (out_len) *out_len = total;
  if (total > out_cap) {
    set_err("gzip_encode: output needs %zu bytes, out_cap %zu", total, out_cap);
    return B200Z_E_NOSPC;
  }
  // header (_gzip_encoder_web.dart:77-90): magic, deflate, flags 0, MTIME, XFL 0, OS 255
  size_t o = 0;
  out[o++] = 0x1f; out[o++] = 0x8b; out[o++] = 8; out[o++] = 0;
  for (int i = 0; i < 4; ++i) out[o++] = (uint8_t)(mtime >> (8 * i));
  out[o++] = 0; out[o++] = 255;
  if (n) CU(cudaMemcpyAsync(out + o, g.d_out.p, n, cudaMemcpyDeviceToHost, g.stream));
  o += n;
  uint32_t crc;
  rc = device_crc32((const uint8_t *)g.d_in.p, in_len, &crc);
  if (rc) return rc;
  for (int i = 0; i < 4; ++i) out[o++] = (uint8_t)(crc >> (8 * i));
  for (int i = 0; i < 4; ++i) out[o++] = (uint8_t)((uint32_t)in_len >> (8 * i));
  CU(cudaStreamSynchronize(g.stream));
  return B200Z_OK;
}

size_t b200z_gzip_bound(const uint8_t *in, size_t in_len) {
  size_t total = 0;
  return hinted_run(in, in_len, 0, nullptr, &total) == in_len ? total : 0;  // every member hinted, or unknown
}

int b200z_gzip_decode(const uint8_t *in, size_t in_len, int verify, uint8_t *out, size_t out_cap, size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  size_t pos = 0, out_pos = 0, needed = 0;
  rc = gzip_fast_path(in, in_len, out, out_cap, &pos, &out_pos, &needed);
  if (rc) {
    if (out_len) *out_len = needed;
    return rc;
  }
  size_t n = out_pos;
  if (pos < in_len) {
    // whatever the hinted run did not cover (no hints, a lying hint, the zlib fall-back): generic path
    const size_t done_out = out_pos;
    rc = stage_input(in, in_len);
    if (rc) return rc;
    rc = gzip_decode_staged(in, in_len, verify, out_cap, &n, pos, out_pos);
    if (out_len) *out_len = n;
    if (rc == B200Z_E_NOSPC || rc == B200Z_E_NODEVICE) return rc;
    size_t hi = n > out_cap ? out_cap : n;
    if (hi > done_out)
      CU(cudaMemcpyAsync(out + done_out, (uint8_t *)g.d_out.p + done_out, hi - done_out, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    return rc;
  }
  if (out_len) *out_len = n;
  return B200Z_OK;
}

int b200z_zlib_decode(const uint8_t *in, size_t in_len, int verify, int raw, uint8_t *out, size_t out_cap,
                      size_t *out_len) {
  int rc = require_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g.mu);
  CU(cudaSetDevice(g.device));
  rc = stage_input(in, in_len);
  if (rc) return rc;
  size_t n = 0;
  rc = zlib_decode_staged(in, in_len, 0, verify, raw, /*big_endian=*/1, 0, out_cap, &n);
  if (out_len) *out_len = n;
  if (rc == B200Z_E_NOSPC || rc == B200Z_E_NODEVICE) return rc;
  if (n > out_cap) n = out_cap;
  if (n) CU(cudaMemcpyAsync(out, g.d_out.p, n, cudaMemcpyDeviceToHost, g.stream));
  CU(cudaStreamSynchronize(g.stream));
  return rc;
}

}  // extern "C"
