// b200z_multi.cu -- several GPUs of one box driven by ONE process (SURVEY.md 8b: the `device_mask` of b200z_init and the
// `n_gpus` of the batch entry points; 8e: independent units are dealt to the GPUs, nothing else is exchanged).
//
// The reference decodes the members of a gzip stream in one loop (lib/src/codecs/zlib/_gzip_decoder_web.dart:27-38) and
// returns one buffer.  Here the members (or the units of a batch) are cut into one contiguous range per GPU, balanced by
// compressed bytes; every GPU gets its range over its own PCIe link, decodes it with the same kernels as the single-GPU
// path (launch_inflate) and writes its part of the output stream straight to its place in the caller's buffer.  With
// B200Z_MULTI_GATHER the shards are also exchanged over NVLink (NCCL, one grouped broadcast per shard -- an all-gather of
// unequal pieces) so that afterwards EVERY device holds the whole stream in block order: that is the form a consumer on
// the device wants (b200z_multi_device_output).  NCCL is looked up at run time (dlopen): the library has no link-time
// dependency on it, and without B200Z_MULTI_GATHER it is never touched.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "b200z_internal.h"

#ifndef B200Z_EMU
#include <dlfcn.h>
#endif

namespace b200z {
namespace {

struct Buf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    const size_t want = n + (n >> 3) + 4096;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      p = nullptr;
      return e;
    }
    cap = want;
    return cudaSuccess;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct Dev {
  int device = -1;
  cudaStream_t s = nullptr;
  Buf in, out, ws, meta;
  void *h_meta = nullptr;  // pinned: results of this device's units
  size_t h_meta_cap = 0;
  void *comm = nullptr;    // ncclComm_t
};

struct Multi {
  std::mutex mu;
  bool inited = false;
  std::vector<Dev> devs;
  bool nccl_tried = false, nccl_ok = false;
  size_t full_bytes = 0;  // size of the gathered stream of the last B200Z_MULTI_GATHER call
};
Multi M;

// ---- NCCL by name (nccl.h is not needed to build: the few types used are spelled out) ----
typedef int (*nccl_init_all_t)(void **comms, int ndev, const int *devlist);
typedef int (*nccl_destroy_t)(void *comm);
typedef int (*nccl_group_t)(void);
typedef int (*nccl_bcast_t)(const void *send, void *recv, size_t count, int dtype, int root, void *comm, cudaStream_t s);
typedef const char *(*nccl_errstr_t)(int);
struct Nccl {
  void *lib = nullptr;
  nccl_init_all_t init_all = nullptr;
  nccl_destroy_t destroy = nullptr;
  nccl_group_t group_start = nullptr, group_end = nullptr;
  nccl_bcast_t bcast = nullptr;
  nccl_errstr_t errstr = nullptr;
} N;
const int kNcclUint8 = 1;  // ncclUint8 (nccl.h: ncclInt8 = 0, ncclUint8 = 1)

bool nccl_load() {
#ifdef B200Z_EMU
  return false;
#else
  if (N.lib) return true;
  const char *names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char *nm : names) {
    N.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (N.lib) break;
  }
  if (!N.lib) return false;
  N.init_all = (nccl_init_all_t)dlsym(N.lib, "ncclCommInitAll");
  N.destroy = (nccl_destroy_t)dlsym(N.lib, "ncclCommDestroy");
  N.group_start = (nccl_group_t)dlsym(N.lib, "ncclGroupStart");
  N.group_end = (nccl_group_t)dlsym(N.lib, "ncclGroupEnd");
  N.bcast = (nccl_bcast_t)dlsym(N.lib, "ncclBroadcast");
  N.errstr = (nccl_errstr_t)dlsym(N.lib, "ncclGetErrorString");
  if (!N.init_all || !N.destroy || !N.group_start || !N.group_end || !N.bcast) {
    N.lib = nullptr;
    return false;
  }
  return true;
#endif
}

char m_err[400];
#define MCU(x)                                                                                      \
  do {                                                                                              \
    cudaError_t e__ = (x);                                                                          \
    if (e__ != cudaSuccess) {                                                                       \
      snprintf(m_err, sizeof m_err, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(e__), __FILE__, __LINE__); \
      set_error_text(m_err);                                                                        \
      return B200Z_E_NODEVICE;                                                                      \
    }                                                                                               \
  } while (0)

struct Share {  // what one device does in a call
  size_t u0 = 0, u1 = 0;        // its units [u0, u1)
  uint64_t in_lo = 0, in_hi = 0;  // the input bytes they cover
  uint64_t out_lo = 0, out_hi = 0;
};

// The units are cut into one contiguous range per device, balanced by compressed bytes.
std::vector<Share> deal(const uint64_t *in_off, const uint32_t *in_len, const uint64_t *out_off, const uint32_t *out_cap,
                        size_t n, size_t ndev) {
  std::vector<Share> sh(ndev);
  uint64_t total = 0;
  for (size_t u = 0; u < n; ++u) total += in_len[u];
  size_t u = 0;
  uint64_t acc = 0;
  for (size_t d = 0; d < ndev; ++d) {
    sh[d].u0 = u;
    const uint64_t want = total * (d + 1) / ndev;
    while (u < n && (acc < want || d + 1 == ndev)) acc += in_len[u++];
    sh[d].u1 = u;
    uint64_t ilo = ~0ull, ihi = 0, olo = ~0ull, ohi = 0;
    for (size_t k = sh[d].u0; k < sh[d].u1; ++k) {
      ilo = std::min<uint64_t>(ilo, in_off[k]);
      ihi = std::max<uint64_t>(ihi, in_off[k] + in_len[k]);
      olo = std::min<uint64_t>(olo, out_off[k]);
      ohi = std::max<uint64_t>(ohi, out_off[k] + out_cap[k]);
    }
    if (sh[d].u1 == sh[d].u0) ilo = ihi = olo = ohi = 0;
    sh[d].in_lo = ilo;
    sh[d].in_hi = ihi;
    sh[d].out_lo = olo;
    sh[d].out_hi = ohi;
  }
  return sh;
}

// Decodes the units on the devices of M.  Host buffers; results in the caller's arrays.  gather: every device also
// receives the other devices' shards (the devices' output buffers then all hold [0, out_bytes)).
int batch_multi(const uint8_t *in_base, const uint64_t *in_off, const uint32_t *in_len, uint8_t *out_base, size_t out_bytes,
                const uint64_t *out_off, const uint32_t *out_cap, uint32_t *out_len, int32_t *status, uint32_t *in_used, size_t n,
                bool gather) {
  const size_t ndev = M.devs.size();
  std::vector<Share> sh = deal(in_off, in_len, out_off, out_cap, n, ndev);
  if (gather) {
    if (!M.nccl_tried) {
      M.nccl_tried = true;
      if (nccl_load()) {
        std::vector<void *> comms(ndev, nullptr);
        std::vector<int> ids(ndev);
        for (size_t d = 0; d < ndev; ++d) ids[d] = M.devs[d].device;
        const int rc = N.init_all(comms.data(), (int)ndev, ids.data());
        if (rc == 0) {
          for (size_t d = 0; d < ndev; ++d) M.devs[d].comm = comms[d];
          M.nccl_ok = true;
        } else {
          snprintf(m_err, sizeof m_err, "ncclCommInitAll failed: %s", N.errstr ? N.errstr(rc) : "?");
          set_error_text(m_err);
        }
      } else {
        set_error_text("B200Z_MULTI_GATHER: libnccl.so.2 not found");
      }
    }
    if (!M.nccl_ok) return B200Z_E_NODEVICE;
  }
  // ---- every device: its input range in, kernels, its output range out -- all asynchronous, one stream per device ----
  for (size_t d = 0; d < ndev; ++d) {
    Dev &dv = M.devs[d];
    const Share &s = sh[d];
    const size_t nu = s.u1 - s.u0;
    MCU(cudaSetDevice(dv.device));
    if (gather) MCU(dv.out.reserve(out_bytes + 64));
    if (nu == 0) continue;
    const size_t in_bytes = (size_t)(s.in_hi - s.in_lo), ob = (size_t)(s.out_hi - s.out_lo);
    MCU(dv.in.reserve(in_bytes + 64));
    if (!gather) MCU(dv.out.reserve(ob + 64));
    const size_t mb = nu * 36 + 256;  // in_off, out_off (u64) + in_len, out_cap, out_len, status, in_used (u32)
    MCU(dv.meta.reserve(mb));
    if (dv.h_meta_cap < mb) {
      if (dv.h_meta) cudaFreeHost(dv.h_meta);
      dv.h_meta = nullptr;
      dv.h_meta_cap = 0;
      MCU(cudaHostAlloc(&dv.h_meta, mb + (mb >> 2), cudaHostAllocDefault));
      dv.h_meta_cap = mb + (mb >> 2);
    }
    uint8_t *hm = (uint8_t *)dv.h_meta, *dm = (uint8_t *)dv.meta.p;
    uint64_t *h_io = (uint64_t *)hm, *h_oo = h_io + nu;
    uint32_t *h_il = (uint32_t *)(h_oo + nu), *h_oc = h_il + nu;
    uint8_t *d_out = (uint8_t *)dv.out.p + (gather ? (size_t)s.out_lo : 0);  // gathered: the final position in the full stream
    for (size_t k = 0; k < nu; ++k) {
      h_io[k] = in_off[s.u0 + k] - s.in_lo;
      h_oo[k] = out_off[s.u0 + k] - s.out_lo;
      h_il[k] = in_len[s.u0 + k];
      h_oc[k] = out_cap[s.u0 + k];
    }
    MCU(cudaMemcpyAsync(dm, hm, nu * 24, cudaMemcpyHostToDevice, dv.s));
    MCU(cudaMemcpyAsync(dv.in.p, in_base + s.in_lo, in_bytes, cudaMemcpyHostToDevice, dv.s));
    const size_t wsb = inflate_ws_bytes(nu, ob);
    MCU(dv.ws.reserve(wsb));
    InflateBatch b;
    b.in_base = (const uint8_t *)dv.in.p;
    b.in_off = (const uint64_t *)dm;
    b.out_off = (const uint64_t *)dm + nu;
    b.in_len = (const uint32_t *)(dm + nu * 16);
    b.out_cap = b.in_len + nu;
    b.out_len = (uint32_t *)(dm + nu * 24);
    b.status = (int32_t *)(b.out_len + nu);
    b.in_used = b.out_len + 2 * nu;
    b.out_base = d_out;
    b.n_units = nu;
    b.ws = inflate_ws_carve(dv.ws.p, nu, ob);
    MCU(launch_inflate(b, dv.s));
    MCU(cudaMemcpyAsync(hm + nu * 24, dm + nu * 24, nu * 12, cudaMemcpyDeviceToHost, dv.s));
    // the device's slots only, not its min..max envelope: the bytes between slots (or other devices' slots inside the
    // envelope when out_off is not monotone) are not this device's to write
    if (!gather && ob) MCU(copy_slots_to_host(out_base, d_out, s.out_lo, out_off + s.u0, out_cap + s.u0, nu, dv.s));
  }
#ifndef B200Z_EMU
  if (gather) {
    // every shard goes from its owner to everybody: one grouped set of broadcasts == an all-gather of unequal pieces
    // over NVLink.  Each device's stream carries its part, behind its own decode.
    int rc = N.group_start();
    for (size_t r = 0; r < ndev && rc == 0; ++r) {
      const size_t bytes = (size_t)(sh[r].out_hi - sh[r].out_lo);
      if (bytes == 0) continue;
      for (size_t d = 0; d < ndev && rc == 0; ++d) {
        uint8_t *p = (uint8_t *)M.devs[d].out.p + sh[r].out_lo;
        rc = N.bcast(p, p, bytes, kNcclUint8, (int)r, M.devs[d].comm, M.devs[d].s);
      }
    }
    const int rc2 = N.group_end();
    if (rc || rc2) {
      snprintf(m_err, sizeof m_err, "NCCL broadcast failed: %s", N.errstr ? N.errstr(rc ? rc : rc2) : "?");
      set_error_text(m_err);
      return B200Z_E_NODEVICE;
    }
    M.full_bytes = out_bytes;
    // the host gets every shard once, from its owner
    for (size_t d = 0; d < ndev; ++d) {
      const size_t ob = (size_t)(sh[d].out_hi - sh[d].out_lo);
      if (!ob) continue;
      MCU(cudaSetDevice(M.devs[d].device));
      MCU(cudaMemcpyAsync(out_base + sh[d].out_lo, (uint8_t *)M.devs[d].out.p + sh[d].out_lo, ob, cudaMemcpyDeviceToHost, M.devs[d].s));
    }
  }
#endif
  for (size_t d = 0; d < ndev; ++d) {
    Dev &dv = M.devs[d];
    MCU(cudaSetDevice(dv.device));
    MCU(cudaStreamSynchronize(dv.s));
    const size_t nu = sh[d].u1 - sh[d].u0;
    if (!nu) continue;
    const uint32_t *r = (const uint32_t *)((uint8_t *)dv.h_meta + nu * 24);
    memcpy(out_len + sh[d].u0, r, nu * 4);
    memcpy(status + sh[d].u0, r + nu, nu * 4);
    memcpy(in_used + sh[d].u0, r + 2 * nu, nu * 4);
  }
  return B200Z_OK;
}

}  // namespace
}  // namespace b200z

using namespace b200z;

extern "C" {

int b200z_multi_init(uint32_t device_mask, uint32_t flags) {
  (void)flags;
  std::lock_guard<std::mutex> lk(M.mu);
  if (M.inited) return B200Z_OK;
  const int n = b200z_device_count();
  std::vector<int> ids;
  for (int d = 0; d < 32; ++d)
    if ((device_mask >> d) & 1u) {
      if (d >= n) {
        snprintf(m_err, sizeof m_err, "b200z_multi_init: CUDA device %d not available (%d visible): there is no CPU fallback", d, n);
        set_error_text(m_err);
        return B200Z_E_NODEVICE;
      }
      ids.push_back(d);
    }
  if (ids.empty()) {
    set_error_text("b200z_multi_init: empty device mask");
    return n > 0 ? B200Z_E_ARG : B200Z_E_NODEVICE;
  }
  // the single-device entry points (framing fall-backs) run on the first device of the mask
  const int rc = b200z_init(ids[0], 0);
  if (rc) return rc;
  M.devs.resize(ids.size());
  for (size_t i = 0; i < ids.size(); ++i) {
    M.devs[i].device = ids[i];
    MCU(cudaSetDevice(ids[i]));
    MCU(cudaStreamCreateWithFlags(&M.devs[i].s, cudaStreamNonBlocking));
  }
  MCU(cudaSetDevice(ids[0]));
  M.inited = true;
  return B200Z_OK;
}

int b200z_multi_device_count(void) { return M.inited ? (int)M.devs.size() : 0; }

void b200z_multi_shutdown(void) {
  std::lock_guard<std::mutex> lk(M.mu);
  if (!M.inited) return;
  for (Dev &d : M.devs) {
    cudaSetDevice(d.device);
    cudaStreamSynchronize(d.s);
#ifndef B200Z_EMU
    if (d.comm && N.destroy) N.destroy(d.comm);
#endif
    d.in.release(); d.out.release(); d.ws.release(); d.meta.release();
    if (d.h_meta) cudaFreeHost(d.h_meta);
    cudaStreamDestroy(d.s);
  }
  cudaSetDevice(M.devs[0].device);
  M.devs.clear();
  M.inited = false;
  M.nccl_tried = M.nccl_ok = false;
}

const void *b200z_multi_device_output(int slot, size_t *bytes) {
  if (bytes) *bytes = 0;
  if (!M.inited || slot < 0 || (size_t)slot >= M.devs.size() || M.full_bytes == 0) return nullptr;
  if (bytes) *bytes = M.full_bytes;
  return M.devs[slot].out.p;
}

int b200z_inflate_batch_multi(const uint8_t *in_base, size_t in_bytes, const uint64_t *in_off, const uint32_t *in_len,
                              uint8_t *out_base, size_t out_bytes, const uint64_t *out_off, const uint32_t *out_cap,
                              uint32_t *out_len, int32_t *status, uint32_t *in_used, size_t n_units, uint32_t flags) {
  if (!M.inited) {
    set_error_text("b200z_multi_init has not been called (or no CUDA device): there is no CPU fallback");
    return B200Z_E_NODEVICE;
  }
  if (n_units == 0) return B200Z_OK;
  for (size_t u = 0; u < n_units; ++u)
    if (in_off[u] > in_bytes || in_len[u] > in_bytes - in_off[u] || out_off[u] > out_bytes || out_cap[u] > out_bytes - out_off[u]) {
      snprintf(m_err, sizeof m_err, "inflate_batch_multi: unit %zu exceeds the buffers", u);
      set_error_text(m_err);
      return B200Z_E_ARG;
    }
  std::lock_guard<std::mutex> lk(M.mu);
  M.full_bytes = 0;
  return batch_multi(in_base, in_off, in_len, out_base, out_bytes, out_off, out_cap, out_len, status, in_used, n_units,
                     (flags & B200Z_MULTI_GATHER) != 0);
}

// GZipDecoderWeb().decodeBytes over the devices of b200z_multi_init: the run of members that carry size hints is dealt to
// the devices; whatever is left (no hints, a hint that lied, the zlib fall-back) goes through b200z_gzip_decode's
// member-by-member path on the first device -- the same bytes either way.
int b200z_gzip_decode_multi(const uint8_t *in, size_t in_len, int verify, uint8_t *out, size_t out_cap, size_t *out_len,
                            uint32_t flags) {
  if (!M.inited) {
    set_error_text("b200z_multi_init has not been called (or no CUDA device): there is no CPU fallback");
    return B200Z_E_NODEVICE;
  }
  std::vector<HintedMember> ms;
  size_t promised = 0;
  const size_t end = gzip_hinted_members(in, in_len, 0, &ms, &promised);
  if (ms.empty() || end != in_len || promised > out_cap) return b200z_gzip_decode(in, in_len, verify, out, out_cap, out_len);
  const size_t n = ms.size();
  std::vector<uint64_t> io(n), oo(n);
  std::vector<uint32_t> il(n), oc(n), ol(n), us(n);
  std::vector<int32_t> st(n);
  size_t o = 0;
  for (size_t i = 0; i < n; ++i) {
    io[i] = ms[i].hdr_end;
    il[i] = (uint32_t)(ms[i].next - ms[i].hdr_end);
    oo[i] = o;
    oc[i] = ms[i].isize;
    o += ms[i].isize;
  }
  int rc;
  {
    std::lock_guard<std::mutex> lk(M.mu);
    M.full_bytes = 0;
    rc = batch_multi(in, io.data(), il.data(), out, o, oo.data(), oc.data(), ol.data(), st.data(), us.data(), n,
                     (flags & B200Z_MULTI_GATHER) != 0);
  }
  if (rc) return rc;
  for (size_t i = 0; i < n; ++i)
    if (!(st[i] == B200Z_U_DONE && ol[i] == ms[i].isize && ms[i].hdr_end + us[i] + 8 == ms[i].next))
      return b200z_gzip_decode(in, in_len, verify, out, out_cap, out_len);  // a hint was not exact: the careful way
  if (out_len) *out_len = o;
  return B200Z_OK;
}

}  // extern "C"
