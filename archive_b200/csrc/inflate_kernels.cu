// inflate_kernels.cu -- sm_100a DEFLATE decode for batches of independent raw DEFLATE streams.
//
// Replaces (reference, paths relative to /root/reference/):
//   lib/src/codecs/zlib/inflate.dart:104-401   Inflate._inflate/_parseBlock/_parseDynamicHuffmanBlock/
//                                              _decodeHuffman/_decode/_readBits/_readCodeByTable
//   lib/src/codecs/zlib/_huffman_table.dart:9-46  HuffmanTable
//   lib/src/util/output_memory_stream.dart:41-98  writeByte / writeBackReference
//
// Two kernels (DESIGN.md "K1"):
//   k_inflate_decode  lane-per-stream: every lane of a warp walks its OWN stream in SIMT lockstep
//                     (table lookup -> shift -> next lookup is a serial chain per stream, so the
//                     only data parallelism is across streams).  Per-lane Huffman LUTs live in shared
//                     memory; the compressed bytes are read through L1 in aligned 32-bit words.  The
//                     output of this phase is a TOKEN stream per unit (literal / match / stored-run),
//                     not bytes: resolving LZ77 copies needs the warp, not a lane.
//   k_inflate_expand  warp-per-stream: turns tokens into bytes.  32 tokens -> warp prefix sum of
//                     lengths -> every lane owns ONE OUTPUT BYTE of a 32-byte window, finds its token
//                     by a shuffle binary search, and resolves out[p] = out[p - dist] (chasing through
//                     bytes of the same window that are not written yet).
#ifdef B200Z_EMU  // CPU emulation build (tests/host_emul/inflate_emul.cpp): kernels only
#include "cuda_emu.h"
alignas(16) static uint32_t cuemu_dyn_smem[64 * 1024];
#define B200Z_DECODE_THREADS 32
#define B200Z_EXPAND_THREADS 256
namespace b200z {
struct InflateWs {
  uint32_t *tokens = nullptr, *htokens = nullptr;
  size_t hstride = 0;
  uint32_t *pieces = nullptr;
  uint8_t *uscratch = nullptr;
  uint32_t hist = 0;
};
}  // namespace b200z
#else
#include "b200z_internal.h"
#endif
#include "inflate_decode.cuh"
#include "inflate_fast.cuh"

#include <stdlib.h>

#include <vector>

namespace b200z {

// ---------------------------------------------------------------------------------------------
// phase 1
// ---------------------------------------------------------------------------------------------
#ifdef B200Z_EMU
#define B200Z_LDCS(p) (*(p))
#define B200Z_DYN_SMEM(name) uint32_t *name = cuemu_dyn_smem
#else
#define B200Z_LDCS(p) __ldcs(p)
#define B200Z_DYN_SMEM(name) extern __shared__ __align__(16) uint32_t name[]
#endif

// HIST: the unit may reach InflateWs::hist bytes of earlier output (single gzip members decoded behind their predecessors).
// The batch kernels are the HIST = false instantiations: the history term folds away and their code is what it was.
template <bool HIST>
__global__ void __launch_bounds__(B200Z_DECODE_THREADS)
k_inflate_decode(const uint8_t *__restrict__ in_base, const uint64_t *__restrict__ in_off,
                 const uint32_t *__restrict__ in_len, const uint64_t *__restrict__ out_off,
                 const uint32_t *__restrict__ out_cap, InflateWs ws, uint32_t *__restrict__ out_len,
                 int32_t *__restrict__ status, uint32_t *__restrict__ in_used, uint32_t n_units, int units_per_warp,
                 int lanes_per_unit, int count_only, int after_fast) {
  B200Z_DYN_SMEM(smem);
  uint16_t *s_len_tab = reinterpret_cast<uint16_t *>(smem);
  uint32_t *s_dist_tab = smem + 16;
  uint32_t *s_xtab = smem + 48;  // [0,32) length symbols, [32,64) distance symbols: (base << 4) | extra_bits
  for (int i = threadIdx.x; i < 32; i += blockDim.x) {
    s_len_tab[i] = c_len_tab[i];
    s_dist_tab[i] = c_dist_tab[i];
    s_xtab[i] = c_len_tab[i];
    s_xtab[32 + i] = c_dist_tab[i];
  }
  __syncthreads();

  const int lane = threadIdx.x & 31;
  const int warp_in_block = threadIdx.x >> 5;
  const uint32_t gwarp = blockIdx.x * (blockDim.x >> 5) + warp_in_block;
  // a stream owns lanes_per_unit consecutive lanes: the first decodes it exactly, the others are its speculative
  // helpers (inflate_decode.cuh).  Every lane stays in the decode loop (it votes once per turn so the warp
  // reconverges); lanes without a stream are born finished.
  const int sidx = lane / lanes_per_unit, sub = lane % lanes_per_unit;
  const uint32_t unit = gwarp * units_per_warp + sidx;
  // after_fast: k_inflate_fast has been over the batch; a unit it finished carries 1 in word 1 of its piece table
  const bool active = sidx < units_per_warp && unit < n_units &&
                      !(after_fast && ws.pieces[(size_t)unit * PIECE_WORDS + 1] == 1u);

  uint16_t *lut_l = reinterpret_cast<uint16_t *>(smem + CONST_WORDS +
                                                 (warp_in_block * units_per_warp + (active ? sidx : 0)) * LANE_STRIDE_WORDS);
  uint16_t *lut_d = lut_l + (1 << LBITS);
  // (16-byte aligned: the slots are read back with one 128-bit load)
  uint32_t *s_stage = smem + ((CONST_WORDS + (blockDim.x >> 5) * units_per_warp * LANE_STRIDE_WORDS + 3) & ~3) + warp_in_block * STAGE_WORDS;

  SpecCtx sc;
  sc.lane = lane;
  sc.sub = sub;
  sc.G = lanes_per_unit;
  sc.stage = s_stage + lane * 4;
  sc.spec = lanes_per_unit > 1 && ws.htokens != nullptr && !count_only;
  sc.count_only = count_only != 0;
  sc.hplane = nullptr;
  sc.hstride = ws.hstride;
  sc.hcap = 0;
  sc.bm = nullptr;
  sc.pieces = nullptr;
  sc.hist = HIST ? ws.hist : 0u;
  uint32_t *tok = nullptr;
  if (active) {
    const uint64_t oo = out_off[unit];
    const uint32_t cap = out_cap[unit];
    tok = ws.tokens + oo;  // token region mirrors the output layout (<= 1 token per output byte)
    if (lanes_per_unit > 1 && ws.htokens && !count_only) {
      sc.hplane = ws.htokens + (oo >> SPEC_HSHIFT);
      sc.hcap = (uint32_t)(((oo + cap) >> SPEC_HSHIFT) - (oo >> SPEC_HSHIFT));
    }
    uint8_t *us = ws.uscratch + (size_t)unit * USCRATCH_BYTES;
    sc.bm = reinterpret_cast<uint32_t *>(us);
    sc.pieces = count_only ? nullptr : ws.pieces + (size_t)unit * PIECE_WORDS;
  }
  const UnitResult r = inflate_decode_unit(active, active ? in_base + in_off[unit] : nullptr, active ? in_len[unit] : 0u,
                                           active ? out_cap[unit] : 0u, tok, lut_l, lut_d, s_len_tab, s_dist_tab, s_xtab, sc);
  if (!active || sub != 0) return;
  out_len[unit] = r.out_len;
  status[unit] = r.status;
  in_used[unit] = r.in_used;
}

// ---------------------------------------------------------------------------------------------
// phase 2
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t tok_len(uint32_t t, bool payload) {
  if (payload) return 0;
  if (t & TOK_LIT) return 1;
  if (t & TOK_STORED) return t & 0xffff;
  return t >> 16;
}

template <bool HIST>
__global__ void __launch_bounds__(B200Z_EXPAND_THREADS)
k_inflate_expand(InflateWs ws, const uint8_t *__restrict__ in_base, const uint64_t *__restrict__ in_off, uint8_t *out_base,
                 const uint64_t *__restrict__ out_off, const uint32_t *__restrict__ out_cap, uint32_t *__restrict__ out_len,
                 int32_t *__restrict__ status, uint32_t n_units, int after_fast) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t unit = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; unit < n_units; unit += warps) {
    if (after_fast && ws.pieces[(size_t)unit * PIECE_WORDS + 1] == 1u) continue;  // finished by k_inflate_fast
    const uint64_t oo = out_off[unit];
    // Positions below count from `hist` bytes in front of the unit (InflateWs::hist; 0 unless the unit is a gzip member
    // decoded on its own behind its predecessors): the range check, the capacity check and the source reads then need
    // nothing extra.
    const uint32_t hist = HIST ? ws.hist : 0u;
    const uint32_t cap = HIST ? (out_cap[unit] > 0xffffffffu - hist ? 0xffffffffu : out_cap[unit] + hist) : out_cap[unit];
    const uint32_t *P = ws.pieces + (size_t)unit * PIECE_WORDS;
    const uint32_t np = P[0];
    uint8_t *out = out_base + oo - hist;
    const uint8_t *in = in_base + in_off[unit];
    uint32_t pos0 = hist;
    bool stop = false;
    for (uint32_t pi = 0; pi < np && !stop; ++pi) {
      const uint32_t src = P[2 + 3 * pi], pstart = P[3 + 3 * pi], nt = P[4 + 3 * pi];
      const uint32_t *T = (src == 0 ? ws.tokens + oo : ws.htokens + (size_t)(src - 1) * ws.hstride + (oo >> SPEC_HSHIFT)) + pstart;
    for (uint32_t g = 0; g < nt && !stop; g += 32) {
      uint32_t t = (g + lane < nt) ? B200Z_LDCS(T + g + lane) : 0u;  // read once: do not keep it in L2
      uint32_t tprev = __shfl_up_sync(FULL, t, 1);
      const bool payload = lane > 0 && (tprev >> 30) == 1u;  // payload words have top bits 00: no chains
      uint32_t len = tok_len(t, payload);
      // inclusive prefix sum of lengths
      uint32_t incl = len;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        uint32_t v = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += v;
      }
      const bool is_stored = !payload && (t & 0xC0000000u) == TOK_STORED;
      // Range checks of the reference, here because tokens adopted from helper lanes were decoded without knowing
      // their absolute position: a back-reference before the start of the output throws (output_memory_stream.dart:
      // 83-86), output beyond the caller's capacity is B200Z_U_NOSPC.  The unit ends with the last good token.
      {
        const bool is_match = !payload && len != 0u && (t & 0xC0000000u) == 0u;
        const bool bad_range = is_match && (t & 0xffffu) > pos0 + (incl - len);
        const bool bad_cap = len != 0u && pos0 + incl > cap;
        const unsigned bad = __ballot_sync(FULL, bad_range || bad_cap);
        if (bad) {
          const int fb = __ffs((int)bad) - 1;
          const bool r_range = __shfl_sync(FULL, (int)bad_range, fb) != 0;
          if (lane >= fb) {
            t = 0;
            len = 0;
          }
          incl = len;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            uint32_t v = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += v;
          }
          stop = true;
          const uint32_t good = __shfl_sync(FULL, incl, 31);
          if (lane == 0) {
            status[unit] = r_range ? B200Z_U_RANGE : B200Z_U_NOSPC;
            out_len[unit] = pos0 + good - hist;
          }
        }
      }
      const uint32_t total = __shfl_sync(FULL, incl, 31);
      const uint32_t start = incl - len;  // relative to pos0
      unsigned stored_mask = __ballot_sync(FULL, is_stored && len != 0u);

      if (stored_mask == 0) {
        // ---- byte-parallel windows ----
        for (uint32_t w = 0; w < total; w += 32) {
          const uint32_t p = w + lane;
          const bool active = p < total;
          // The token of byte q of this window = (tokens that start before the window) + (tokens that start inside it at
          // or before q) - 1: one vote and one OR-reduction per window instead of a binary search per byte.  (Tokens of
          // length 0 only trail the real ones in a group that takes this path, so rank == lane.)
          const uint32_t before = (uint32_t)__popc(__ballot_sync(FULL, len != 0u && start < w));
          const uint32_t starts = __reduce_or_sync(FULL, (len != 0u && start >= w && start < w + 32u) ? (1u << (start - w)) : 0u);
          int j = (int)(before + (uint32_t)__popc(starts & ((2u << lane) - 1u))) - 1;
          j &= 31;
          uint32_t tj = __shfl_sync(FULL, t, j);
          uint32_t sj = __shfl_sync(FULL, start, j);
          bool have = !active || (tj & TOK_LIT);
          uint32_t byte = tj & 0xff;
          int src2 = 0;
          if (!have) {
            uint32_t dist = tj & 0xffff;
            src2 = (int)p - (int)dist;
            if (src2 >= (int)sj) {  // overlapping run: fold whole periods back before the match
              int k = (src2 - (int)sj) / (int)dist + 1;
              src2 -= k * (int)dist;
            }
          }
          // chase sources that are still inside this (unwritten) window
          while (__any_sync(FULL, !have && src2 >= (int)w)) {
            const bool need = !have && src2 >= (int)w;
            uint32_t q = need ? (uint32_t)src2 : w;
            int j2 = (int)(before + (uint32_t)__popc(starts & ((2u << (q - w)) - 1u))) - 1;  // w <= q < w + 32
            j2 &= 31;
            uint32_t t2 = __shfl_sync(FULL, t, j2);
            uint32_t s2 = __shfl_sync(FULL, start, j2);
            if (need) {
              if (t2 & TOK_LIT) {
                byte = t2 & 0xff;
                have = true;
              } else {
                uint32_t d2 = t2 & 0xffff;
                src2 = (int)q - (int)d2;
                if (src2 >= (int)s2) {
                  int k = (src2 - (int)s2) / (int)d2 + 1;
                  src2 -= k * (int)d2;
                }
              }
            }
          }
          if (active) {
            if (!have) byte = out[(long long)pos0 + src2];
            out[pos0 + p] = (uint8_t)byte;
          }
          __syncwarp();
        }
      } else {
        // ---- rare: group holds a stored run -> walk the 32 tokens in order, warp-cooperatively ----
        for (int i = 0; i < 32; ++i) {
          uint32_t ti = __shfl_sync(FULL, t, i);
          uint32_t li = __shfl_sync(FULL, len, i);
          uint32_t si = __shfl_sync(FULL, start, i);
          uint32_t nx = __shfl_sync(FULL, t, (i + 1) & 31);
          if (li == 0) continue;
          uint8_t *dst = out + pos0 + si;
          if (ti & TOK_LIT) {
            if (lane == 0) dst[0] = (uint8_t)ti;
          } else if ((stored_mask >> i) & 1u) {
            const uint8_t *srcp = in + (((size_t)((ti >> 16) & 3u) << 30) | nx);
            for (uint32_t b = lane; b < li; b += 32) dst[b] = srcp[b];
          } else {
            uint32_t dist = ti & 0xffff;
            const uint8_t *srcp = dst - dist;
            if (dist >= li) {
              for (uint32_t b = lane; b < li; b += 32) dst[b] = srcp[b];
            } else {
              for (uint32_t b = lane; b < li; b += 32) dst[b] = srcp[b % dist];
            }
          }
          __syncwarp();
        }
      }
      pos0 += total;
    }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Flush points: positions right after every byte-aligned 00 00 FF FF (the empty stored block Z_SYNC_FLUSH / Z_FULL_FLUSH
// leave behind).  Candidates only: the caller proves them by decoding (b200z_api.cu, zip members).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_find_flush_markers(const uint8_t *__restrict__ in, unsigned long long n, unsigned long long *__restrict__ list,
                     uint32_t *__restrict__ count, uint32_t cap) {
  const unsigned long long i0 = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 16ull;
  if (i0 >= n) return;
  uint8_t b[19];
  for (int k = 0; k < 19; ++k) b[k] = (i0 + k < n) ? in[i0 + k] : (uint8_t)0x55;
  for (int k = 0; k < 16; ++k)
    if (b[k] == 0 && b[k + 1] == 0 && b[k + 2] == 0xff && b[k + 3] == 0xff && i0 + k + 4 <= n) {
      uint32_t slot = atomicAdd(count, 1u);
      if (slot < cap) list[slot] = i0 + k + 4;
    }
}

#ifndef B200Z_EMU
// ---------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------
static int g_num_sms = 0;

// optional per-kernel timing (CUDA events on the launching stream; bench.py's roofline breakdown)
struct ProfTriple { cudaEvent_t a, f, b, c; };  // start, after k_inflate_fast, after k_inflate_decode, after k_inflate_expand
static bool g_prof = false;
static std::vector<ProfTriple> g_prof_events;
void profile_enable(bool on) { g_prof = on; }
int profile_read(double *fast_ms, double *decode_ms, double *expand_ms, uint64_t *n) {
  *fast_ms = *decode_ms = *expand_ms = 0;
  *n = 0;
  for (auto &t : g_prof_events) {
    if (cudaEventSynchronize(t.c) != cudaSuccess) return -1;
    float f = 0, d = 0, e = 0;
    cudaEventElapsedTime(&f, t.a, t.f);
    cudaEventElapsedTime(&d, t.f, t.b);
    cudaEventElapsedTime(&e, t.b, t.c);
    *fast_ms += f;
    *decode_ms += d;
    *expand_ms += e;
    ++*n;
    cudaEventDestroy(t.a); cudaEventDestroy(t.f); cudaEventDestroy(t.b); cudaEventDestroy(t.c);
  }
  g_prof_events.clear();
  return 0;
}

size_t inflate_ws_bytes(size_t n_units, size_t extent) {
  const size_t tok = (extent * 4 + 511) & ~(size_t)255;
  const size_t hstride = (extent >> SPEC_HSHIFT) + 64;
  const size_t hb = ((SPEC_MAX_G - 1) * hstride * 4 + 255) & ~(size_t)255;
  const size_t pb = (n_units * PIECE_WORDS * 4 + 255) & ~(size_t)255;
  const size_t ub = (n_units * (size_t)USCRATCH_BYTES + 255) & ~(size_t)255;
  return tok + hb + pb + ub + 256;
}
size_t inflate_ws_extent_for(size_t n_units, size_t bytes) {
  const size_t fixed = inflate_ws_bytes(n_units, 0) + 1024;
  if (bytes <= fixed) return 0;
  return (bytes - fixed) / (4 + (SPEC_MAX_G - 1)) ;
}
InflateWs inflate_ws_carve(void *ws, size_t n_units, size_t extent) {
  InflateWs w;
  uint8_t *p = reinterpret_cast<uint8_t *>(ws);
  const size_t tok = (extent * 4 + 511) & ~(size_t)255;
  w.hstride = (extent >> SPEC_HSHIFT) + 64;
  const size_t hb = ((SPEC_MAX_G - 1) * w.hstride * 4 + 255) & ~(size_t)255;
  const size_t pb = (n_units * PIECE_WORDS * 4 + 255) & ~(size_t)255;
  w.tokens = reinterpret_cast<uint32_t *>(p);
  w.htokens = reinterpret_cast<uint32_t *>(p + tok);
  w.pieces = reinterpret_cast<uint32_t *>(p + tok + hb);
  w.uscratch = p + tok + hb + pb;
  return w;
}
InflateWs inflate_ws_slice(const InflateWs &w, size_t first_unit, size_t first_out_byte) {
  InflateWs s = w;
  s.tokens = w.tokens + first_out_byte;
  s.htokens = w.htokens + (first_out_byte >> SPEC_HSHIFT);
  s.pieces = w.pieces + first_unit * PIECE_WORDS;
  s.uscratch = w.uscratch + first_unit * (size_t)USCRATCH_BYTES;
  return s;
}

cudaError_t launch_find_markers(const uint8_t *d_in, size_t n, unsigned long long *d_list, uint32_t *d_count, uint32_t cap,
                                cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(d_count, 0, 4, stream);
  if (e != cudaSuccess || n == 0) return e;
  const unsigned long long threads = (n + 15) / 16;
  k_find_flush_markers<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(d_in, n, d_list, d_count, cap);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_inflate(const InflateBatch &b, cudaStream_t stream) {
  if (b.n_units == 0) return cudaSuccess;
  int cur_dev = 0;
  cudaGetDevice(&cur_dev);
  if (!g_num_sms) {
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, cur_dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  // Streams per warp.  Decode is latency-bound per stream, so what matters first is that every
  // scheduler has a warp; beyond that, packing more streams into a warp only saves issue slots.
  const int warps_per_block = B200Z_DECODE_THREADS / 32;
  int upw = 32;
  {
    static int forced = -1;
    if (forced < 0) {
      const char *e = getenv("B200Z_UPW");
      forced = e ? atoi(e) : 0;
    }
    if (forced >= 1 && forced <= 32) {
      upw = forced;
    } else {
      // measured on B200 (profiles/r1_inflate_upw_sweep.md): 8 streams per warp at ~14 warps per SM is the best point for
      // 16 Ki streams -- wider warps are latency-bound (too few warps per scheduler), narrower ones issue-bound
      const uint64_t target_warps = (uint64_t)g_num_sms * 12 / (uint64_t)(b.share > 0 ? b.share : 1);
      while (upw > 1 && (b.n_units + upw - 1) / upw < target_warps) upw >>= 1;
    }
  }
  // lanes per stream: the lanes a warp has left over decode the same streams speculatively (inflate_decode.cuh)
  int lpu = 32 / upw;
  {
    static int forced_g = -1;
    if (forced_g < 0) {
      const char *e = getenv("B200Z_SPEC_G");
      forced_g = e ? atoi(e) : 0;
    }
    if (lpu > SPEC_MAX_G) lpu = SPEC_MAX_G;
    if (forced_g >= 1 && forced_g < lpu) lpu = forced_g;
    while (lpu & (lpu - 1)) lpu &= lpu - 1;
  }
  const uint64_t n_warps = (b.n_units + upw - 1) / upw;
  const unsigned blocks = (unsigned)((n_warps + warps_per_block - 1) / warps_per_block);
  const size_t smem = inflate_decode_smem_bytes(warps_per_block, upw);
  static size_t attr_smem_dev[64] = {};
  size_t &attr_smem = attr_smem_dev[cur_dev & 63];
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(k_inflate_decode<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_inflate_decode<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr_smem = smem;
  }
  ProfTriple pt{};
  if (g_prof) {
    cudaEventCreate(&pt.a); cudaEventCreate(&pt.f); cudaEventCreate(&pt.b); cudaEventCreate(&pt.c);
    cudaEventRecord(pt.a, stream);
  }
  // k_inflate_fast first (inflate_fast.cuh): a CTA per unit, everything in shared memory.  It finishes the clean units
  // whose output fits its window and flags them; the two exact kernels below then only see what is left.
  int after_fast = 0;
  int fast_only = 0;
  {
    // B200Z_FAST=0 (read at every launch, so a process can time both) leaves everything to the exact pair.  Default on:
    // on the benchmark shape the kernel moves a fifth of the pair's DRAM bytes and takes 10.3 ms per GiB whatever the
    // data and the batch size, where the pair takes 9.3 ms on one rank's data and 13.5 on the others', and twice that
    // when a batch is launched in quarters (profiles/r2_summary.md, DESIGN.md K1f).
    // B200Z_FAST=2 is a test and diagnostic mode: k_inflate_fast alone.  The units it leaves keep the out_len / status /
    // in_used the caller put there and their output slots are not written, so a caller can see which units it finished.
    const char *fe = getenv("B200Z_FAST");
    const int fast_on = fe ? atoi(fe) : 1;
    fast_only = fast_on == 2;
    if (fast_on && !b.count_only && b.ws.hist == 0 && b.ws.pieces != nullptr && b.ws.uscratch != nullptr) {
      static uint64_t attr_done = 0;  // one bit per device: function attributes belong to the device's context
      if (!((attr_done >> (cur_dev & 63)) & 1u)) {
        cudaError_t e = cudaFuncSetAttribute(k_inflate_fast, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fp::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        attr_done |= 1ull << (cur_dev & 63);
      }
      // two resident CTAs per SM, each walks its share of the units.  B200Z_FAST_SPARE_SMS leaves SMs to kernels that
      // have to run beside this one -- a collective that forwards the finished chunk while the next one is decoded
      // (persistent CTAs that fill every SM keep NCCL's kernel waiting until the grid drains)
      int spare = 0;
      if (const char *se = getenv("B200Z_FAST_SPARE_SMS")) spare = atoi(se);
      if (spare < 0 || spare >= g_num_sms) spare = 0;
      uint64_t fblocks = (uint64_t)(g_num_sms - spare) * 2u;
      if (fblocks > b.n_units) fblocks = b.n_units;
      // the unit counter: the first word of the exact kernels' scratch, which is dead until they run
      uint32_t *next_unit = reinterpret_cast<uint32_t *>(b.ws.uscratch);
      cudaError_t me = cudaMemsetAsync(next_unit, 0, sizeof(uint32_t), stream);
      if (me != cudaSuccess) return me;
      k_inflate_fast<<<(unsigned)fblocks, fp::NTT, fp::SMEM_BYTES, stream>>>(b.in_base, b.in_off, b.in_len, b.out_base, b.out_off, b.out_cap,
                                                                        b.out_len, b.status, b.in_used, (uint32_t)b.n_units,
                                                                        b.ws.pieces + 1, (uint32_t)PIECE_WORDS, next_unit);
      count_launch();
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) return e;
      after_fast = 1;
    }
  }
  if (g_prof) cudaEventRecord(pt.f, stream);
  if (fast_only && after_fast) {
    if (g_prof) {
      cudaEventRecord(pt.b, stream);
      cudaEventRecord(pt.c, stream);
      g_prof_events.push_back(pt);
    }
    return cudaSuccess;
  }
  if (b.ws.hist)
    k_inflate_decode<true><<<blocks, B200Z_DECODE_THREADS, smem, stream>>>(b.in_base, b.in_off, b.in_len, b.out_off, b.out_cap, b.ws,
                                                                         b.out_len, b.status, b.in_used, (uint32_t)b.n_units, upw,
                                                                         b.count_only ? 1 : lpu, b.count_only ? 1 : 0, after_fast);
  else
    k_inflate_decode<false><<<blocks, B200Z_DECODE_THREADS, smem, stream>>>(b.in_base, b.in_off, b.in_len, b.out_off, b.out_cap, b.ws,
                                                                          b.out_len, b.status, b.in_used, (uint32_t)b.n_units, upw,
                                                                          b.count_only ? 1 : lpu, b.count_only ? 1 : 0, after_fast);
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (g_prof) cudaEventRecord(pt.b, stream);
  if (b.count_only) {
    if (g_prof) {
      cudaEventRecord(pt.c, stream);
      g_prof_events.push_back(pt);
    }
    return cudaSuccess;
  }
  const int ewarps = B200Z_EXPAND_THREADS / 32;
  uint64_t eblocks = (b.n_units + ewarps - 1) / ewarps;
  // resident expand warps x 32 KiB of LZ77 window each should stay inside the 126 MB L2
  static int bps = -1;
  if (bps < 0) {
    const char *e = getenv("B200Z_EXPAND_BPS");
    bps = e ? atoi(e) : 0;
    if (bps <= 0) bps = 32;
  }
  const uint64_t max_blocks = (uint64_t)g_num_sms * (uint64_t)bps;
  if (eblocks > max_blocks) eblocks = max_blocks;
  if (b.ws.hist)
    k_inflate_expand<true><<<(unsigned)eblocks, B200Z_EXPAND_THREADS, 0, stream>>>(b.ws, b.in_base, b.in_off, b.out_base, b.out_off,
                                                                                 b.out_cap, b.out_len, b.status, (uint32_t)b.n_units, after_fast);
  else
    k_inflate_expand<false><<<(unsigned)eblocks, B200Z_EXPAND_THREADS, 0, stream>>>(b.ws, b.in_base, b.in_off, b.out_base, b.out_off,
                                                                                  b.out_cap, b.out_len, b.status, (uint32_t)b.n_units, after_fast);
  count_launch();
  if (g_prof) {
    cudaEventRecord(pt.c, stream);
    g_prof_events.push_back(pt);
  }
  return cudaGetLastError();
}
#endif  // !B200Z_EMU

}  // namespace b200z

#ifdef FP_PROF
// FP_PROF builds only (scripts/build_variant.sh prof -DFP_PROF): k_inflate_fast's clocks per phase, summed over CTAs; cleared by the read.
extern "C" int b200z_debug_fast_prof(unsigned long long *out16 /* [20] */) {
  unsigned long long z[20] = {0};
  if (cudaMemcpyFromSymbol(out16, b200z::fp::g_fp_prof, sizeof z) != cudaSuccess) return -1;
  return cudaMemcpyToSymbol(b200z::fp::g_fp_prof, z, sizeof z) == cudaSuccess ? 0 : -1;
}
#endif
