// sweep_types.h — constants, kernel parameter blocks and the launch macros shared by the
// tick kernels (sweep_kernels.cuh), the exchange kernels (gather_kernels.cuh) and the host
// runtime (sweep.cu, gather.cu).  No kernel definitions here: both .cu files include it.
#pragma once
#ifndef AMSWEEP_EMULATE  // tests/emu compiles these files for the CPU (cuda_emu.h supplies the model)
#include <cuda_runtime.h>
#endif
#include <stddef.h>
#include <stdint.h>

#include "../../include/amsweep.h"
#include "civil.h"
#include "tz_eval.h"

// Kernel launches are spelled through two macros so that tests/emu can compile the host
// runtime (sweep.cu) for the CPU emulator as well.  AM_LAUNCH is the plain <<<>>> launch;
// AM_LAUNCH_PDL adds the programmatic-stream-serialization attribute (programmatic dependent
// launch): the kernel may be scheduled while its predecessor in the stream drains and calls
// pdl_wait() (griddepcontrol.wait) before it touches anything the predecessor wrote — the
// launch latency between the four small kernels of a tick disappears behind the sweep's tail.
#ifndef AM_LAUNCH
#ifndef AMSWEEP_EMULATE
#define AM_LAUNCH(kernel, grid, block, stream, ...) kernel<<<(grid), (block), 0, (stream)>>>(__VA_ARGS__)
#define AM_LAUNCH_PDL(kernel, grid, block, strm_, ...)                                    \
  do {                                                                                    \
    cudaLaunchConfig_t _cfg = {};                                                         \
    _cfg.gridDim = dim3(grid);                                                            \
    _cfg.blockDim = dim3(block);                                                          \
    _cfg.stream = (strm_);                                                                \
    cudaLaunchAttribute _at[1];                                                           \
    _at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                       \
    _at[0].val.programmaticStreamSerializationAllowed = 1;                                \
    _cfg.attrs = _at;                                                                     \
    _cfg.numAttrs = 1;                                                                    \
    (void)cudaLaunchKernelEx(&_cfg, kernel, __VA_ARGS__);                                 \
  } while (0)
#else
#define AM_LAUNCH(kernel, grid, block, stream, ...) ((void)(stream), emu::launch(kernel, dim3(grid), dim3(block), __VA_ARGS__))
#define AM_LAUNCH_PDL(kernel, grid, block, stream, ...) ((void)(stream), emu::launch(kernel, dim3(grid), dim3(block), __VA_ARGS__))
#endif
#endif
#define AM_SWEEP_KERNEL(closed, masks) sweep_tick_kernel<closed, masks>  // one macro argument
#define AM_BLOCK_KERNEL(closed, lists) sweep_block_kernel<closed, lists>

// The sixteen record columns, in am_record_cols_t member order: position = the column id of
// am_sweep_column_ptr.  am_record_t has a field of the same name and type for each.
#define AM_RECORD_COLUMNS(X)                                                                        \
  X(minute) X(hour) X(dom) X(month) X(dow) X(ras) X(flags) X(finished_at) X(runs_limit) X(reset_interval) \
  X(success) X(failed) X(remedy_success) X(remedy_failed) X(remedy_total) X(remedy_finished_at)

namespace amsweep {

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
constexpr int kRecPerWarp = 128;             // 2 halves x 32 lanes x 2 records
constexpr int kTile = kWarps * kRecPerWarp;  // 1024 records per CTA
constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr int kNumAcc = 16;  // == number of u64 fields of am_tick_stats_t
constexpr int kMaxWorld = 16;

// A "group" is the unit of the list rebuild: 8 tiles = 8192 records = 256 bitmap words = one
// expand CTA with one word per thread.
constexpr int kGroupTiles = 8;
constexpr uint32_t kGroupRecords = kGroupTiles * kTile;  // 8192
constexpr uint32_t kGroupWords = kGroupRecords / 32;     // 256
constexpr uint32_t kTileWords = kTile / 32;              // 32
static_assert(kBlock == 256 && kTile == 1024, "bitmap layout: 32 words per tile, 4 per warp");

// A shard's device columns are the public column set, passed to kernels by value.  Column k is
// the k-th pointer of the struct: the host runtime addresses columns by id through that.
using DevCols = am_record_cols_t;
constexpr int kNumCols = 16;
struct ColumnInfo { size_t offset, elem; };
#define AM_COLUMN_INFO(name) {offsetof(am_record_cols_t, name), sizeof(*am_record_cols_t{}.name)},
constexpr ColumnInfo kColumns[kNumCols] = {AM_RECORD_COLUMNS(AM_COLUMN_INFO)};
#undef AM_COLUMN_INFO
constexpr bool columns_are_a_pointer_array() {
  for (int k = 0; k < kNumCols; ++k)
    if (kColumns[k].offset != k * sizeof(void*)) return false;
  return sizeof(am_record_cols_t) == kNumCols * sizeof(void*);
}
static_assert(columns_are_a_pointer_array(), "am_record_cols_t: sixteen pointers in AM_RECORD_COLUMNS order");

// What one tick of one shard leaves behind for the list rebuild (expand_kernel) and for the
// NVLink exchange: the same four arrays whether they are the sweep's own buffers or the copy
// a peer pushed into this GPU's exchange block.
struct TickOut {
  uint32_t* bitmap;        // [n_groups * 256] bit b of word w = record 32 w + b of the shard is emitted
  uint32_t* group_count;   // [n_groups] emitted records per group (REDs of the tiles; zero on entry)
  uint32_t* group_prefix;  // [n_groups + 1] exclusive prefix of group_count (scan_groups_kernel)
  uint32_t* tile_exc;      // [n_tiles] exceptions per tile
  uint32_t* exc_seg;       // [n_tiles * 1024] per tile: (offset in tile << 8) | action, ascending
};

struct SweepParams {
  DevCols c;
  uint64_t n_records;
  uint64_t shard_base;
  uint64_t seed;
  int64_t T;
  TickWords words;  // T's UTC fields as one-hot words, computed once per tick by the launcher
  uint32_t n_tiles;
  uint32_t mode;
  TickOut out;
  unsigned long long* acc;   // [kNumAcc] statistics accumulators (zero on entry)
  const TickWords* tz_table; // [zones + 1] T's LOCAL fields per registered time zone (entry 0 = UTC), written by
                             // tz_words_kernel ahead of the sweep; NULL when no zone is registered
};

struct ScanParams {
  uint32_t* group_count;        // this tick's per-group sums; zeroed again once read
  uint32_t* group_prefix;       // [n_groups + 1]
  unsigned long long* acc;      // acc[1] = n_emitted
  uint32_t* out_count;          // may be NULL: min(n_emitted, cap) for device-side consumers
  uint32_t n_groups, cap;
};

struct ExpandSrc {
  const uint32_t* bitmap;
  const uint32_t* group_prefix;
  const uint32_t* tile_exc;
  const uint32_t* exc_seg;
  uint64_t base;  // added to the shard-local record number to form the output index
  uint32_t n_groups, n_tiles;
};
struct ExpandParams {
  ExpandSrc src[kMaxWorld];  // rank order; the output is their concatenation
  void* out_idx;             // [cap] u32 or u64
  uint8_t* out_act;          // [cap]
  unsigned long long* acc;   // action-bit counts and index checksums of rank `stats_rank` (may be NULL)
  uint64_t stats_base;       // global index of that rank's record 0 (checksums are over global indices)
  uint64_t cap;
  int world, stats_rank, idx_bytes;
};

}  // namespace amsweep
