// b200z_internal.h -- shared declarations between the kernels and the C-ABI layer (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <vector>

#include "../../include/b200z.h"

#ifndef B200Z_LBITS
#define B200Z_LBITS 9  // literal/length primary LUT bits (2^9 x u16 per stream)
#endif
#ifndef B200Z_DBITS
#define B200Z_DBITS 8  // distance primary LUT bits
#endif
#define B200Z_DECODE_THREADS 32   // one warp per block: finest block-scheduler granularity
#define B200Z_EXPAND_THREADS 256

namespace b200z {

// Device workspace of one inflate batch (inflate_kernels.cu).  `extent` = size of the output layout in bytes.
struct InflateWs {
  uint32_t *tokens = nullptr;   // [extent] u32: unit u's own tokens start at word out_off[u] (<= 1 token per output byte)
  uint32_t *htokens = nullptr;  // 7 helper planes of hstride words: helper k of unit u writes from plane k-1, word out_off[u] >> 2
  size_t hstride = 0;
  uint32_t *pieces = nullptr;   // [n_units][PIECE_WORDS]: which token runs make up the unit, in order
  uint8_t *uscratch = nullptr;  // [n_units][USCRATCH_BYTES]: slow tables + helper boundary bitmaps
  // Bytes of EARLIER output that lie directly in front of a unit's output slot and that its back-references may reach.
  // 0 for independent streams (Inflate(bytes), zip members, zlib streams: each has an output stream of its own).  GZip
  // members share ONE OutputStream in the reference (_gzip_decoder_web.dart:38: Inflate.stream(input, output: output)), so
  // a member's distance may reach into the members before it (output_memory_stream.dart:79-98 checks against the whole
  // stream): the member-by-member path sets this for its single-unit batches.
  uint32_t hist = 0;
};
size_t inflate_ws_bytes(size_t n_units, size_t extent);
size_t inflate_ws_extent_for(size_t n_units, size_t bytes);  // largest extent a workspace of `bytes` serves
InflateWs inflate_ws_carve(void *ws, size_t n_units, size_t extent);
InflateWs inflate_ws_slice(const InflateWs &w, size_t first_unit, size_t first_out_byte);

struct InflateBatch {
  const uint8_t *in_base;
  const uint64_t *in_off;
  const uint32_t *in_len;
  uint8_t *out_base;
  const uint64_t *out_off;
  const uint32_t *out_cap;
  uint32_t *out_len;
  int32_t *status;
  uint32_t *in_used;
  size_t n_units;
  InflateWs ws;
  int share = 1;     // how many batches run concurrently on the device (sizes the streams-per-warp choice)
  bool count_only = false;  // sizes only: out_len / status / in_used, no tokens, no output bytes
};

cudaError_t launch_inflate(const InflateBatch &b, cudaStream_t stream);
// Device-to-host copy of the output slots of n units: host[out_off[u] .. +out_cap[u]) <- dev[out_off[u] - lo ..), one copy per
// run of slots that touch or overlap.  The caller's bytes between slots are not written.
cudaError_t copy_slots_to_host(uint8_t *host, const uint8_t *dev, uint64_t lo, const uint64_t *out_off, const uint32_t *out_cap,
                               size_t n, cudaStream_t stream);
cudaError_t launch_find_markers(const uint8_t *d_in, size_t n, unsigned long long *d_list, uint32_t *d_count, uint32_t cap,
                                cudaStream_t stream);

// ---- BZip2 (bzip2_kernels.cu) ----
struct Bz2Entropy {  // K7, one warp per candidate block
  const uint32_t *words;
  uint64_t n_bytes;
  const unsigned long long *blk_bit;  // bit position of each candidate's 48-bit magic
  uint32_t n_blocks, nblock_max;
  uint32_t *rec_val, *rec_pos;  // [n_blocks][nblock_max]
  uint32_t *n_rec, *nblock, *orig_ptr, *randomised;
  unsigned long long *end_bit;
  int32_t *status;
  uint32_t *fast_flag = nullptr;  // [n_blocks], may be null: 1 = the block was decoded by k_bz2_entropy_fast
  uint8_t *sym8 = nullptr;        // [n_blocks][nblock_max]: K8's byte array, by candidate slot (the fast kernel writes it)
};
struct Bz2Ibwt {  // K8 over the validated chain
  const void *chain;  // BzChain[n_chain] (device)
  uint32_t n_chain, nblock_max;
  const uint32_t *rec_val, *rec_pos;
  uint8_t *sym8;    // [n_chain][nblock_max]
  uint32_t *chist;  // [n_chain][chunks_max][256]
  uint32_t *tt;     // [n_chain][nblock_max]
  uint32_t *seg_len, *seg_next, *seg_off;  // [n_chain][4098]
  uint32_t *seg_resume;                    // [n_chain][4098]: where the walk of a segment stood when its slot was full
  uint8_t *slots;                          // [n_chain][4098][bz2_slot_bytes_per_block() / 4098]: a segment's bytes before they are placed
  uint32_t *walk_ctr;                      // [2]: the work counters of k_bz2_walk_len / k_bz2_walk_emit
  int32_t *irregular;                      // [n_chain]
  uint32_t *cycle_len;                     // [n_chain]
  uint8_t *raw;                            // [n_chain][nblock_max]
  uint32_t *slice_state, *slice_out;       // [n_chain][1024]
  unsigned long long *block_out, *block_off;  // [n_chain], [n_chain + 1]
  uint32_t *block_crc;                         // [n_chain]
  uint8_t *out;
  unsigned long long out_cap;
  bool any_randomised = false;
  bool carry_off = false;  // block_off[0] already holds the first block's offset (bz2_launch_ibwt_group)
  bool any_records = true; // some block of the chain comes with records (the exact kernels'; long runs of the fast one)
  int phase = 0;           // 0: all of K8; 1: everything up to the blocks' output offsets; 2: the RLE1 output pass only
};
struct BzChainHost {
  uint32_t cand, nblock, n_rec, orig_ptr;
  uint32_t flags;  // bit 0: randomised block (serial path in K8)
};
size_t bz2_entropy_smem();
cudaError_t bz2_launch_scan(const uint8_t *d_in, uint64_t n_bytes, unsigned long long *d_cand, uint32_t *d_ncand,
                            uint32_t cap, cudaStream_t s);
cudaError_t bz2_launch_entropy(const Bz2Entropy &a, cudaStream_t s);
// blocks K7 left with status -3 (a damaged block that the reference keeps decoding): d_list = their indices into a's arrays
cudaError_t bz2_launch_entropy_literal(const Bz2Entropy &a, const uint32_t *d_list, uint32_t n_list, cudaStream_t s);
size_t bz2_slot_bytes_per_block();
cudaError_t bz2_launch_ibwt(const Bz2Ibwt &a, cudaStream_t s);
cudaError_t bz2_launch_ibwt_group(const Bz2Ibwt &a, uint32_t lo, uint32_t hi, cudaStream_t s);
void count_launch();
void profile_enable(bool on);
int profile_read(double *fast_ms, double *decode_ms, double *expand_ms, uint64_t *n);

// ---- file streams (b200z_file.cu) and the hooks it uses (b200z_api.cu) ----
void set_error_text(const char *msg);  // b200z_last_error() text of the calling thread
size_t gzip_hinted_prefix(const uint8_t *in, size_t n, size_t *out_bytes);
struct HintedMember {
  size_t hdr_end, next;  // first byte of the DEFLATE stream; first byte behind the member
  uint32_t isize;
};
// the run of members from `pos` on that carry the BGZF 'BC' size and a believable ISIZE (b200z_api.cu: hinted_run)
size_t gzip_hinted_members(const uint8_t *in, size_t n, size_t pos, std::vector<HintedMember> *ms, size_t *out_bytes);
int gzip_decode_hinted(const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *in_used, size_t *out_len);
int gzip_decode_after(const uint8_t *in, size_t n, int verify, const uint8_t *hist, size_t hist_len, uint8_t *out, size_t out_cap,
                      size_t *out_len);
void file_release();  // frees the pinned segment buffers (b200z_shutdown)

// ---- Deflate (deflate_kernels.cu) ----
struct DeflStoredBlock {
  uint32_t start, len, eof;
};
size_t deflate_bound(size_t n);
// levels 1-3 over a batch (k_defl_fast_batch): where one member's bytes are and where its tokens go (device pointers;
// tok / tally_ss / next_ss hold n + 2 words each)
struct DeflFastMember {
  const uint8_t *d = nullptr;
  uint32_t n = 0, pad_ = 0;
  uint32_t *tok = nullptr, *tally_ss = nullptr, *next_ss = nullptr, *ntok = nullptr;
};
cudaError_t deflate_fast_tokens_batch(const DeflFastMember *d_list, uint32_t n_mem, int level, int window_bits, uint32_t *d_counter,
                                      cudaStream_t s);
size_t deflate_workspace_bytes(size_t n);
cudaError_t deflate_slow_device(const uint8_t *d_in, size_t n, int level, int window_bits, uint8_t *d_out, size_t out_cap,
                                void *ws, size_t ws_bytes, size_t *out_len, uint32_t *stats, cudaStream_t s, const DeflFastMember *pre = nullptr);
cudaError_t deflate_stored_device(const uint8_t *d_in, const DeflStoredBlock *h_blocks, uint32_t n_blocks, uint8_t *d_out,
                                  size_t out_cap, void *ws, size_t ws_bytes, size_t *out_len, cudaStream_t s);
cudaError_t crc32_tiles_device(const uint8_t *d_in, size_t n, uint32_t tile, uint32_t *d_part, cudaStream_t s);

}  // namespace b200z
