// Host orchestration + C-ABI entry points of the occupancy -> SignedDistanceField path (sm_100a).
// Device code: edt_scan_registers.cuh / edt_device.cuh (z scan, finalize helpers),
// edt_envelope_window.cuh (the strided passes) and edt_envelope_lean.cuh (the stack kernel behind
// it). DESIGN.md has the roofline of each kernel.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "common.cuh"
#include "host_transfer.cuh"
#include "edt_device.cuh"
#include "edt_envelope_lean.cuh"
#include "edt_envelope_window.cuh"
#include "edt_scan_registers.cuh"
#include "edt_cells.cuh"
#include "edt_transform.cuh"

namespace vgt_b200
{
namespace edt
{
namespace
{
inline int64_t Square(int64_t v) { return v * v; }

// ------------------------------------------------------------------------------------------------
// Kernel launchers
// ------------------------------------------------------------------------------------------------
template <typename In>
int LaunchScan(const In* d_in, uint32_t* d_out, int64_t num_lines, int32_t length,
               int unknown_is_filled, cudaStream_t stream)
{
  const int num_words = (length + 31) >> 5;
  const size_t smem = sizeof(uint32_t) * 5 * num_words * kScanWarpsPerBlock;
  const int64_t blocks = (num_lines + kScanWarpsPerBlock - 1) / kScanWarpsPerBlock;
  // 128-bit path: every line must start 16-byte aligned in both buffers.
  using Source = typename std::conditional<
      std::is_same<In, float>::value, Float4Source,
      typename std::conditional<std::is_same<In, ObjectSlot>::value, SlotEquals4Source,
                                Uchar4Source>::type>::type;
  const bool aligned = (length % 4 == 0)
      && (reinterpret_cast<uintptr_t>(d_in) % sizeof(typename Source::Vector) == 0)
      && (reinterpret_cast<uintptr_t>(d_out) % sizeof(uint4) == 0);
  if (aligned && length <= 2048)
  {
    // whole line in registers: 1, 2, 4, 8 or 16 iterations of 128 voxels
    const auto launch = [&](auto kernel)
    {
      kernel<<<static_cast<unsigned>(blocks), kScanWarpsPerBlock * kWarp, 0, stream>>>(
          reinterpret_cast<const typename Source::Vector*>(d_in), reinterpret_cast<uint4*>(d_out),
          num_lines, length, unknown_is_filled); NoteKernelLaunch();
    };
    if (length <= 128)
    {
      launch(ScanContiguousAxisRegistersKernel<Source, 1>);
    }
    else if (length <= 256)
    {
      launch(ScanContiguousAxisRegistersKernel<Source, 2>);
    }
    else if (length <= 512)
    {
      launch(ScanContiguousAxisRegistersKernel<Source, 4>);
    }
    else if (length <= 1024)
    {
      launch(ScanContiguousAxisRegistersKernel<Source, 8>);
    }
    else
    {
      launch(ScanContiguousAxisRegistersKernel<Source, 16>);
    }
    VGT_CUDA_TRY(cudaGetLastError(), "ScanContiguousAxisRegistersKernel launch");
    return VGT_B200_OK;
  }
  if (aligned)
  {
    ScanContiguousAxisVec4Kernel<Source>
        <<<static_cast<unsigned>(blocks), kScanWarpsPerBlock * kWarp, smem, stream>>>(
            reinterpret_cast<const typename Source::Vector*>(d_in),
            reinterpret_cast<uint4*>(d_out), num_lines, length, unknown_is_filled); NoteKernelLaunch();
    VGT_CUDA_TRY(cudaGetLastError(), "ScanContiguousAxisVec4Kernel launch");
    return VGT_B200_OK;
  }
  ScanContiguousAxisKernel<In><<<static_cast<unsigned>(blocks), kScanWarpsPerBlock * kWarp, smem,
                                 stream>>>(d_in, d_out, num_lines, length, unknown_is_filled); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "ScanContiguousAxisKernel launch");
  return VGT_B200_OK;
}

// SM count of the current device (148 on B200), cached per host thread.
inline int64_t MultiprocessorCount()
{
  static thread_local int cached_device = -1;
  static thread_local int cached_count = 148;
  int device = 0;
  if (cudaGetDevice(&device) == cudaSuccess && device != cached_device)
  {
    int count = 0;
    if (cudaDeviceGetAttribute(&count, cudaDevAttrMultiProcessorCount, device) == cudaSuccess
        && count > 0)
    {
      cached_count = count;
      cached_device = device;
    }
  }
  return cached_count;
}

template <int kMode, bool kNarrow, bool kSend, bool kBorder, bool kSplit>
int LaunchEnvelopeLeanKernel(uint32_t* d_in, typename OutputOf<kMode>::Type* d_out,
                             uint16_t* d_positions, const LineFamily& family,
                             const FinalizeParams& finalize,
                             typename OutputOf<kMode>::Key* d_keys, cudaStream_t stream,
                             const uint32_t* d_redo_list)
{
  const int64_t tiles = ((family.inner_count + kWarp - 1) / kWarp) * family.num_outer;
  const int64_t blocks = (tiles + kLineWarpsPerBlock - 1) / kLineWarpsPerBlock;
  const int64_t lines = family.num_outer * family.inner_count;
  if (blocks > 0x7fffffffLL || lines * 4 > 0xffffffffLL)
  {
    return FailInvalid("grid too large for one launch");
  }
  // class words + run-end table of every line (6 bytes per 32 voxels), stream-ordered
  StreamScratch<uint32_t> class_scratch;
  VGT_CUDA_TRY(class_scratch.Allocate(
                   static_cast<int64_t>((LeanScratchBytes(family.length, lines) + 3) / 4), stream),
               "envelope class-word scratch");
  LineFamily derived = family;
  derived.stride_bytes = static_cast<uint32_t>(family.line_stride * 4);
  derived.out_stride_bytes = static_cast<uint32_t>(
      family.line_stride * static_cast<int64_t>(sizeof(typename OutputOf<kMode>::Type)));
  derived.last_row = static_cast<uint32_t>(family.length - 1);
  derived.num_words = static_cast<uint32_t>((family.length + 31) >> 5);
  const auto launch = [&](auto kernel)
  {
    kernel<<<static_cast<unsigned>(blocks), kLineWarpsPerBlock * kWarp, 0, stream>>>(
        d_in, d_out, d_positions, class_scratch.get(), derived, finalize, d_keys, d_redo_list); NoteKernelLaunch();
  };
  if constexpr (kMode == kEmitPacked)
  {
    // 16 blocks per SM (32 registers) only when that saves a whole wave over 12 (40 registers)
    const int64_t sms = MultiprocessorCount();
    const int64_t waves_at_16 = (blocks + sms * 16 - 1) / (sms * 16);
    const int64_t waves_at_12 = (blocks + sms * 12 - 1) / (sms * 12);
    if (waves_at_16 == 1 && waves_at_12 > 1)
    {
      launch(EnvelopeAxisLeanKernel<kMode, kNarrow, kSend, kBorder, kSplit, 16>);
    }
    else
    {
      launch(EnvelopeAxisLeanKernel<kMode, kNarrow, kSend, kBorder, kSplit, 12>);
    }
  }
  else
  {
    launch(EnvelopeAxisLeanKernel<kMode, kNarrow, kSend, kBorder, kSplit, 8>);
  }
  VGT_CUDA_TRY(cudaGetLastError(), "EnvelopeAxisLeanKernel launch");
  return VGT_B200_OK;
}

// Send-layout output exists only for the packed intermediate, the virtual border only for the
// finalizing pass, so each mode instantiates two of the four flag combinations.
template <int kMode, bool kNarrow, bool kSplit>
int LaunchEnvelopeLean(uint32_t* d_in, typename OutputOf<kMode>::Type* d_out,
                       uint16_t* d_positions, const LineFamily& family,
                       const FinalizeParams& finalize, typename OutputOf<kMode>::Key* d_keys,
                       cudaStream_t stream, const uint32_t* d_redo_list)
{
  if constexpr (kMode == kEmitPacked)
  {
    if (family.out_parts > 0)
    {
      return LaunchEnvelopeLeanKernel<kMode, kNarrow, true, false, kSplit>(
          d_in, d_out, d_positions, family, finalize, d_keys, stream, d_redo_list);
    }
    return LaunchEnvelopeLeanKernel<kMode, kNarrow, false, false, kSplit>(
        d_in, d_out, d_positions, family, finalize, d_keys, stream, d_redo_list);
  }
  else
  {
    if (family.out_parts > 0)
    {
      return FailInvalid("send layout is only available for the packed intermediate");
    }
    if (finalize.add_virtual_border != 0)
    {
      return LaunchEnvelopeLeanKernel<kMode, kNarrow, false, true, kSplit>(
          d_in, d_out, d_positions, family, finalize, d_keys, stream, d_redo_list);
    }
    return LaunchEnvelopeLeanKernel<kMode, kNarrow, false, false, kSplit>(
        d_in, d_out, d_positions, family, finalize, d_keys, stream, d_redo_list);
  }
}

// A/B switches of the strided passes, for experiments and for the tests that force each route.
// The environment is read ONCE, at the first SDF call of the process; vgt_b200_reload_tuning()
// re-reads it (tests flip the variables inside one process). Snapshots are immutable and never
// freed (a reload leaks one small struct), so concurrent calls read them without locking.
//   VGT_B200_ENVELOPE=lean        the stack kernel alone, no window kernel in front of it
//   VGT_B200_WINDOW_BUDGET=<pct>  joint-search rounds a warp may spend per row of its tile before
//                                 it hands the tile to the stack kernel, in percent (2400 = 24
//                                 per row on average; 0 = never search beyond the registers)
//   VGT_B200_WINDOW_PILOT=0       no pilot launch in front of the window kernel
//   VGT_B200_WINDOW_STAGE=0|1|2   rows ahead by plain loads / through shared memory with per-lane
//                                 cp.async / with cp.async.bulk (TMA engine) + mbarrier
//   VGT_B200_WINDOW_RADIUS_Y=8|10|12  register-window radius of the plain y pass
struct Tuning
{
  bool window_enabled = true;
  uint32_t step_rate = 2400u * 128u / 100u;
  bool pilot = true;
  int stage = -1;      // -1: each pass its measured best
  int radius_y = 0;    // 0: the default
  int blocks_per_sm = 192;  // window kernel: blocks per multiprocessor the segmenting aims at
};

inline const Tuning* LoadTuning()
{
  Tuning* tuning = new Tuning();
  const char* envelope = std::getenv("VGT_B200_ENVELOPE");
  tuning->window_enabled = !(envelope != nullptr && std::strcmp(envelope, "lean") == 0);
  if (const char* budget = std::getenv("VGT_B200_WINDOW_BUDGET"))
  {
    // (capped so that rate x rows of the longest segment stays inside 32 bits)
    const long percent = std::strtol(budget, nullptr, 10);
    tuning->step_rate =
        static_cast<uint32_t>(std::min(std::max(0L, percent), 100000L) * 128 / 100);
  }
  const char* pilot = std::getenv("VGT_B200_WINDOW_PILOT");
  tuning->pilot = !(pilot != nullptr && std::strcmp(pilot, "0") == 0);
  const char* stage = std::getenv("VGT_B200_WINDOW_STAGE");
  if (stage != nullptr && (std::strcmp(stage, "0") == 0 || std::strcmp(stage, "1") == 0
                           || std::strcmp(stage, "2") == 0))
  {
    tuning->stage = stage[0] - '0';
  }
  if (const char* radius = std::getenv("VGT_B200_WINDOW_RADIUS_Y"))
  {
    tuning->radius_y = std::atoi(radius);
  }
  if (const char* blocks = std::getenv("VGT_B200_WINDOW_BLOCKS_PER_SM"))
  {
    tuning->blocks_per_sm = std::min(std::max(std::atoi(blocks), 1), 4096);
  }
  return tuning;
}

std::atomic<const Tuning*> g_tuning{nullptr};

inline const Tuning& CurrentTuning()
{
  const Tuning* tuning = g_tuning.load(std::memory_order_acquire);
  if (tuning == nullptr)
  {
    const Tuning* loaded = LoadTuning();
    if (g_tuning.compare_exchange_strong(tuning, loaded, std::memory_order_acq_rel))
    {
      return *loaded;
    }
    delete loaded;  // another thread was first
    return *tuning;
  }
  return *tuning;
}

// Largest finite partial squared distance the lean kernel's 32-bit sentinels leave room for
// (heights h = f + v^2 must stay well below kNoSiteHeight = 2^30 - 1). Every grid whose axes fit
// VGT_B200_MAX_AXIS stays below it: 2 * 8191^2 < 2^28.
constexpr int64_t kLeanMaxInput = (int64_t{1} << 29) - 1;

// Measurement aid (vgt_b200_sdf_f32_dev_profile): events right around the main window-kernel
// launch of each strided pass, so that the kernel's own duration can be told apart from the
// pass (pilot + decision + window kernel + stack kernel over the redo list). Thread-local: only
// the calling thread's launches are marked.
struct WindowKernelMarks
{
  cudaEvent_t begin[2];
  cudaEvent_t end[2];
  int launches = 0;
};
thread_local WindowKernelMarks* g_window_marks = nullptr;

// The window kernel over every tile of the family; tiles it gives up on are appended to
// d_redo_list (layout in edt_envelope_window.cuh; header and flags zeroed here). With enough tiles
// a pilot launch goes first: it probes two chunks of rows out of every 256 of every 8th tile
// and decides, on the device, whether the window kernel runs at all. On maps with large
// open spaces nearly every tile would end up with the stack kernel anyway, and the window
// kernel's searches would only be wasted.
template <int kMode>
int LaunchEnvelopeWindow(const uint32_t* d_in, typename OutputOf<kMode>::Type* d_out,
                         const LineFamily& family, const FinalizeParams& finalize,
                         typename OutputOf<kMode>::Key* d_keys, uint32_t* d_redo_list,
                         cudaStream_t stream)
{
  const int64_t tiles = ((family.inner_count + kWarp - 1) / kWarp) * family.num_outer;
  const int64_t blocks = (tiles + kWindowWarpsPerBlock - 1) / kWindowWarpsPerBlock;
  if (blocks > 0x7fffffffLL)
  {
    return FailInvalid("grid too large for one launch");
  }
  VGT_CUDA_TRY(cudaMemsetAsync(d_redo_list, 0, sizeof(uint32_t) * kRedoList, stream),
               "redo list reset");
  VGT_CUDA_TRY(cudaMemsetAsync(d_redo_list + kRedoList + tiles, 0, sizeof(uint32_t) * tiles,
                               stream),
               "redo flags reset");
  LineFamily derived = family;
  derived.stride_bytes = static_cast<uint32_t>(family.line_stride * 4);
  derived.out_stride_bytes = static_cast<uint32_t>(
      family.line_stride * static_cast<int64_t>(sizeof(typename OutputOf<kMode>::Type)));
  derived.last_row = static_cast<uint32_t>(family.length - 1);
  derived.num_words = static_cast<uint32_t>((family.length + 31) >> 5);
  const Tuning& tuning = CurrentTuning();
  const uint32_t step_rate = tuning.step_rate;
  // Lines are cut into segments so that there are about six waves of blocks (and never
  // segments shorter than eight chunks; measured at 512^3: 1.68 ms with one segment per line,
  // 1.49 ms with four): the block scheduler then balances tiles of uneven depth
  // and the last wave is thin. A segment re-reads 2 R rows of its neighbours.
  constexpr int kRadius = (kMode == kEmitPacked) ? kWindowRadiusPacked : kWindowRadiusFinal;
  // Rows reach the registers by plain loads one chunk ahead (stage 0, the default of both
  // passes), or through shared memory two chunks ahead: by per-lane cp.async (stage 1), or filled
  // by the TMA engine with one cp.async.bulk per row and an mbarrier per buffer (stage 2; needs
  // rows that start 16-byte aligned and full tiles, else it falls back to stage 1). Measured at
  // 512^3 with the up-front absorb of round 2 (profiles/r2_experiments.md): x pass 0.442 / 0.457
  // / 0.510 ms, y pass 0.413 / 0.431 / 0.476 ms for stage 0 / 1 / 2 - the passes are bound by
  // the alu pipe, not by how the rows arrive, and the staged variants add shared-memory reads
  // and waits. VGT_B200_WINDOW_STAGE=0 / 1 / 2 forces a variant for both passes.
  const bool bulk_ok = family.inner_count % kWarp == 0 && family.line_stride % 4 == 0
      && family.outer_stride % 4 == 0 && reinterpret_cast<uintptr_t>(d_in) % 16 == 0;
  int stage_mode = tuning.stage >= 0 ? tuning.stage : 0;
  if (stage_mode == 2 && !bulk_ok)
  {
    stage_mode = 1;
  }
  const bool staged = stage_mode != 0;
  // (experiment knob: the radius of the plain, unstaged y pass)
  int radius = kRadius;
  if (kMode == kEmitPacked && family.out_parts == 0 && !staged
      && (tuning.radius_y == 8 || tuning.radius_y == 10))
  {
    radius = tuning.radius_y;
  }
  const int64_t chunks = (family.length + radius - 1) / radius;
  const int64_t wanted_blocks =
      static_cast<int64_t>(MultiprocessorCount()) * tuning.blocks_per_sm / kWindowWarpsPerBlock;
  int64_t segments = (wanted_blocks + blocks - 1) / blocks;
  segments = std::max<int64_t>(1, std::min<int64_t>(segments, chunks / 8));
  const int segment_rows = static_cast<int>((chunks + segments - 1) / segments) * radius;
  segments = (family.length + segment_rows - 1) / segment_rows;
  derived.first_segment = 0;
  if (family.out_parts > 1 && family.scatter_base[0] != nullptr)
  {
    // first row of the part after this rank's own
    const int64_t next_part = (family.scatter_rank + 1) % family.out_parts;
    const int64_t wide = family.out_base + 1;
    const int64_t row = next_part < family.out_extra
        ? next_part * wide
        : family.out_extra * wide + (next_part - family.out_extra) * family.out_base;
    derived.first_segment = static_cast<uint32_t>((row / segment_rows) % segments);
  }
  // (VGT_B200_WINDOW_PILOT=0: no pilot, the window kernel works on every tile)
  const bool pilot = tiles >= 16 * static_cast<int64_t>(kPilotStride) && tuning.pilot;
  // (pilot_kernel: the variant that runs the probe launch. In the probe every lane reads the
  // family's last column - it stores nothing and only counts search effort -, which the bulk
  // variant cannot do: its rows arrive as whole tiles. Its probe runs on the cp.async variant.)
  const auto launch_with_pilot = [&](auto kernel, auto pilot_kernel)
  {
    const dim3 threads(kWindowWarpsPerBlock * kWarp);
    WindowKernelMarks* const marks =
        (g_window_marks != nullptr && g_window_marks->launches < 2) ? g_window_marks : nullptr;
    if (!pilot)
    {
      if (marks != nullptr) { cudaEventRecord(marks->begin[marks->launches], stream); }
      kernel<<<dim3(static_cast<unsigned>(blocks), static_cast<unsigned>(segments)), threads, 0,
               stream>>>(d_in, d_out, derived, finalize, d_keys, d_redo_list, step_rate,
                         segment_rows, segment_rows, kSelectAll); NoteKernelLaunch();
      if (marks != nullptr) { cudaEventRecord(marks->end[marks->launches++], stream); }
      return;
    }
    const int64_t pilot_blocks = (blocks + kPilotStride - 1) / kPilotStride;
    const int64_t probes_per_line = (family.length + kPilotSpacing - 1) / kPilotSpacing;
    const int64_t pilot_probes =
        std::min<int64_t>(pilot_blocks * kWindowWarpsPerBlock, tiles) * probes_per_line;
    pilot_kernel<<<dim3(static_cast<unsigned>(pilot_blocks),
                        static_cast<unsigned>(probes_per_line)),
                   threads, 0, stream>>>(d_in, d_out, derived, finalize, d_keys, d_redo_list,
                                   std::min(step_rate, kPilotStepRate), 2 * radius, kPilotSpacing,
                                   kSelectPilot); NoteKernelLaunch();
    DecideWindowModeKernel<<<1, 1, 0, stream>>>(d_redo_list, static_cast<uint32_t>(pilot_probes)); NoteKernelLaunch();
    if (marks != nullptr) { cudaEventRecord(marks->begin[marks->launches], stream); }
    kernel<<<dim3(static_cast<unsigned>(blocks), static_cast<unsigned>(segments)), threads, 0,
             stream>>>(d_in, d_out, derived, finalize, d_keys, d_redo_list, step_rate,
                       segment_rows, segment_rows, kSelectAfterPilot); NoteKernelLaunch();
    if (marks != nullptr) { cudaEventRecord(marks->end[marks->launches++], stream); }
  };
  const auto launch = [&](auto kernel) { launch_with_pilot(kernel, kernel); };
  if constexpr (kMode == kEmitPacked)
  {
    if (family.out_parts > 0)
    {
      launch(EnvelopeAxisWindowKernel<kMode, kWindowRadiusPacked, false, true, kWindowBlocksPacked>);
    }
    else if (stage_mode == 2)
    {
      launch_with_pilot(
          EnvelopeAxisWindowKernel<kMode, kWindowRadiusPacked, false, false, 32, 2>,
          EnvelopeAxisWindowKernel<kMode, kWindowRadiusPacked, false, false, 32, 1>);
    }
    else if (staged)
    {
      launch(EnvelopeAxisWindowKernel<kMode, kWindowRadiusPacked, false, false, 32, 1>);
    }
    else
    {
      if (radius == 8)
      {
        launch(EnvelopeAxisWindowKernel<kMode, 8, false, false, 32>);
      }
      else if (radius == 10)
      {
        launch(EnvelopeAxisWindowKernel<kMode, 10, false, false, 32>);
      }
      else
      {
        launch(EnvelopeAxisWindowKernel<kMode, kWindowRadiusPacked, false, false, kWindowBlocksPacked>);
      }
    }
  }
  else if (family.out_parts > 0)
  {
    return FailInvalid("send layout is only available for the packed intermediate");
  }
  else if (finalize.add_virtual_border != 0)
  {
    if (stage_mode == 2)
    {
      launch_with_pilot(EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, true, false, 32, 2>,
                        EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, true, false, 32, 1>);
    }
    else if (staged)
    {
      launch(EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, true, false, 32, 1>);
    }
    else
    {
      launch(EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, true, false, kWindowBlocksFinal>);
    }
  }
  else if (stage_mode == 2)
  {
    launch_with_pilot(EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, false, false, 32, 2>,
                      EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, false, false, 32, 1>);
  }
  else if (staged)
  {
    launch(EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, false, false, 32, 1>);
  }
  else
  {
    launch(EnvelopeAxisWindowKernel<kMode, kWindowRadiusFinal, false, false, kWindowBlocksFinal>);
  }
  VGT_CUDA_TRY(cudaGetLastError(), "EnvelopeAxisWindowKernel launch");
  return VGT_B200_OK;
}

// One strided-axis pass. d_in is DESTROYED and must not alias d_out.
// max_input: largest finite partial squared distance the pass can see. The window kernel runs
// first and the stack kernel only redoes the tiles it gave up on (short axes with packed 32-bit
// stack entries; longer ones keep the site positions in a stream-ordered uint16 side array).

template <int kMode>
int LaunchEnvelope(uint32_t* d_in, typename OutputOf<kMode>::Type* d_out,
                   const LineFamily& family, int64_t max_input, const FinalizeParams& finalize,
                   typename OutputOf<kMode>::Key* d_keys, cudaStream_t stream)
{
  if (family.length > VGT_B200_MAX_AXIS || max_input > 0x7ffffffeLL)
  {
    return FailInvalid("axis of %d voxels is out of range", family.length);
  }
  const bool packed = family.length <= kInPlaceMaxLength && max_input <= kInPlaceMaxInput;
  if (family.line_stride * 8 > 0xffffffffLL || max_input > kLeanMaxInput)
  {
    // (cannot happen for grids inside VGT_B200_MAX_AXIS: 2 * 8191^2 < 2^28)
    SetLastError("partial distances up to %lld are outside the range of the integer passes",
                 static_cast<long long>(max_input));
    return VGT_B200_ERR_UNSUPPORTED;
  }
  StreamScratch<uint32_t> redo;
  const uint32_t* d_redo_list = nullptr;
  if (CurrentTuning().window_enabled)
  {
    const int64_t tiles = ((family.inner_count + kWarp - 1) / kWarp) * family.num_outer;
    VGT_CUDA_TRY(redo.Allocate(2 * tiles + kRedoList, stream), "envelope redo list");
    const int status = LaunchEnvelopeWindow<kMode>(d_in, d_out, family, finalize, d_keys,
                                                   redo.get(), stream);
    if (status != VGT_B200_OK)
    {
      return status;
    }
    d_redo_list = redo.get();
  }
  if (packed)
  {
    // 32-bit pop test when no product of an h difference and a position difference can overflow.
    const int64_t max_h = max_input + Square(family.length - 1);
    if (max_h * family.length < (int64_t{1} << 31))
    {
      return LaunchEnvelopeLean<kMode, true, false>(d_in, d_out, nullptr, family, finalize,
                                                    d_keys, stream, d_redo_list);
    }
    return LaunchEnvelopeLean<kMode, false, false>(d_in, d_out, nullptr, family, finalize, d_keys,
                                                   stream, d_redo_list);
  }
  // Longer axes / larger distances: site positions go to a stream-ordered uint16 side array
  // (2 bytes per voxel, span = the family's element span).
  const int64_t span = (family.num_outer - 1) * family.outer_stride
      + static_cast<int64_t>(family.length - 1) * family.line_stride + family.inner_count;
  StreamScratch<uint16_t> positions;
  VGT_CUDA_TRY(positions.Allocate(span, stream), "envelope position side array");
  return LaunchEnvelopeLean<kMode, false, true>(d_in, d_out, positions.get(), family, finalize,
                                                d_keys, stream, d_redo_list);
}

struct EventGuard
{
  cudaEvent_t event = nullptr;
  ~EventGuard()
  {
    if (event != nullptr)
    {
      cudaEventDestroy(event);
    }
  }
};

LineFamily FamilyAlongY(int64_t nx, int64_t ny, int64_t nz)
{
  return LineFamily{nx, ny * nz, nz, nz, static_cast<int32_t>(ny)};
}

LineFamily FamilyAlongX(int64_t nx, int64_t ny, int64_t nz)
{
  return LineFamily{1, 0, ny * nz, ny * nz, static_cast<int32_t>(nx)};
}

// z scan then y envelope on an [nx, ny, nz] block; the result lands in d_result. d_other is a
// second buffer of the same size that is used as the intermediate (contents destroyed).
template <typename In>
int RunLocalPasses(const In* d_in, int64_t nx, int64_t ny, int64_t nz, int unknown_is_filled,
                   uint32_t* d_result, uint32_t* d_other, cudaStream_t stream, int send_parts = 0,
                   const uint64_t* scatter_bases = nullptr, int64_t scatter_row_offset = 0,
                   int scatter_rank = 0)
{
  if (send_parts > 1)
  {
    if (send_parts > ny)
    {
      return FailInvalid("more parts (%d) than rows along y (%lld)", send_parts,
                         static_cast<long long>(ny));
    }
    LineFamily family = FamilyAlongY(nx, ny, nz);
    family.out_parts = send_parts;
    family.out_base = static_cast<int32_t>(ny / send_parts);
    family.out_extra = static_cast<int32_t>(ny % send_parts);
    if (scatter_bases == nullptr)
    {
      const int status = LaunchScan<In>(d_in, d_other, nx * ny, static_cast<int32_t>(nz),
                                        unknown_is_filled, stream);
      if (status != VGT_B200_OK)
      {
        return status;
      }
      return LaunchEnvelope<kEmitPacked>(d_other, d_result, family, Square(nz - 1),
                                         FinalizeParams{}, nullptr, stream);
    }
    if (send_parts > 8)
    {
      return FailInvalid("fused exchange supports at most 8 ranks");
    }
    family.scatter_rank = scatter_rank;
    for (int part = 0; part < send_parts; part++)
    {
      family.scatter_base[part] = reinterpret_cast<uint32_t*>(scatter_bases[part]);
    }
    // (Tried: x-chunks with the scan of chunk c + 1 on a second stream under the y pass of chunk
    // c. The y pass fills the register file, so the two kernels only alternate, and the extra
    // pilot / tail per chunk made it slower: 1.57 against 1.45 ms at 2 GPUs.)
    family.scatter_row_offset = scatter_row_offset;
    const int status = LaunchScan<In>(d_in, d_other, nx * ny, static_cast<int32_t>(nz),
                                      unknown_is_filled, stream);
    if (status != VGT_B200_OK)
    {
      return status;
    }
    return LaunchEnvelope<kEmitPacked>(d_other, d_result, family, Square(nz - 1),
                                       FinalizeParams{}, nullptr, stream);
  }
  if (ny <= 1)
  {
    return LaunchScan<In>(d_in, d_result, nx * ny, static_cast<int32_t>(nz), unknown_is_filled,
                          stream);
  }
  const int status = LaunchScan<In>(d_in, d_other, nx * ny, static_cast<int32_t>(nz),
                                    unknown_is_filled, stream);
  if (status != VGT_B200_OK)
  {
    return status;
  }
  return LaunchEnvelope<kEmitPacked>(d_other, d_result, FamilyAlongY(nx, ny, nz), Square(nz - 1),
                                     FinalizeParams{}, nullptr, stream);
}

// Per-call table of finished magnitudes for the finalizing pass (FinalizeParams::magnitude_table):
// every squared distance the grid can produce, capped at 2^20 entries (4 / 8 MB); larger values
// take the direct fp64 path in the kernel.
constexpr int64_t kMagnitudeTableMaxEntries = int64_t{1} << 20;

template <typename Out>
class MagnitudeTable
{
public:
  int Build(int64_t nx, int64_t ny, int64_t nz, double resolution, cudaStream_t stream)
  {
    // (never fewer than kSaturated + 1 entries: the window kernel looks every value it emits up
    // without a bound check, and those are below kSaturated)
    const int64_t largest = std::max<int64_t>(Square(nx - 1) + Square(ny - 1) + Square(nz - 1),
                                              static_cast<int64_t>(kSaturated));
    size_ = static_cast<uint32_t>(std::min(largest + 1, kMagnitudeTableMaxEntries));
    VGT_CUDA_TRY(table_.Allocate(size_, stream), "magnitude table allocation");
    const unsigned threads = 256;
    BuildMagnitudeTableKernel<Out><<<(size_ + threads - 1) / threads, threads, 0, stream>>>(
        table_.get(), size_, resolution); NoteKernelLaunch();
    VGT_CUDA_TRY(cudaGetLastError(), "BuildMagnitudeTableKernel launch");
    return VGT_B200_OK;
  }
  void Attach(FinalizeParams& finalize) const
  {
    finalize.magnitude_table = table_.get();
    finalize.magnitude_table_size = size_;
  }

private:
  StreamScratch<Out> table_;
  uint32_t size_ = 0;
};

// x envelope on an [nx, ny_local, nz] block + finalize. d_packed is destroyed.
template <int kMode>
int RunFinalPass(uint32_t* d_packed, int64_t nx, int64_t ny_local, int64_t nz, int64_t y_offset,
                 int64_t ny_total, double resolution, int add_virtual_border,
                 typename OutputOf<kMode>::Type* d_out, typename OutputOf<kMode>::Type* d_min_max,
                 cudaStream_t stream)
{
  using Out = typename OutputOf<kMode>::Type;
  using Key = typename OutputOf<kMode>::Key;
  StreamScratch<Key> keys;
  if (d_min_max != nullptr)
  {
    VGT_CUDA_TRY(keys.Allocate(2, stream), "min/max scratch");
    ResetMinMaxKeysKernel<Key><<<1, 1, 0, stream>>>(keys.get()); NoteKernelLaunch();
  }
  FinalizeParams finalize{};
  finalize.resolution = resolution;
  finalize.add_virtual_border = add_virtual_border;
  finalize.nx_total = static_cast<int32_t>(nx);
  finalize.ny_total = static_cast<int32_t>(ny_total);
  finalize.nz_total = static_cast<int32_t>(nz);
  finalize.y_offset = static_cast<int32_t>(y_offset);
  finalize.nz = static_cast<int32_t>(nz);
  MagnitudeTable<Out> magnitudes;
  {
    const int built = magnitudes.Build(nx, ny_total, nz, resolution, stream);
    if (built != VGT_B200_OK)
    {
      return built;
    }
    magnitudes.Attach(finalize);
  }
  const int status = LaunchEnvelope<kMode>(d_packed, d_out, FamilyAlongX(nx, ny_local, nz),
                                           Square(nz - 1) + Square(ny_total - 1), finalize,
                                           keys.get(), stream);
  if (status != VGT_B200_OK)
  {
    return status;
  }
  if (d_min_max != nullptr)
  {
    DecodeMinMaxKernel<Out, Key><<<1, 1, 0, stream>>>(keys.get(), d_min_max); NoteKernelLaunch();
    VGT_CUDA_TRY(cudaGetLastError(), "DecodeMinMaxKernel launch");
  }
  return VGT_B200_OK;
}

int CheckSdfArguments(const void* in, const void* out, int64_t nx, int64_t ny, int64_t nz,
                      double resolution)
{
  if (in == nullptr || out == nullptr)
  {
    return FailInvalid("null grid pointer");
  }
  if (!ValidDims(nx, ny, nz))
  {
    return FailInvalid("grid dimensions %lld x %lld x %lld out of range [1, %d]",
                       static_cast<long long>(nx), static_cast<long long>(ny),
                       static_cast<long long>(nz), VGT_B200_MAX_AXIS);
  }
  if (!(resolution > 0.0) || !std::isfinite(resolution))
  {
    return FailInvalid("resolution must be positive and finite");
  }
  return VGT_B200_OK;
}

// The whole path on device-resident data. The output buffer doubles as the first intermediate
// (it is at least 4 bytes per voxel); one stream-ordered scratch of 4 bytes per voxel is the
// second. pass_events: optional 4 events recorded around the three kernels (profiling entry).
template <typename In, int kMode>
int SdfOnDevice(const In* d_in, int64_t nx, int64_t ny, int64_t nz, double resolution,
                int unknown_is_filled, int add_virtual_border,
                typename OutputOf<kMode>::Type* d_sdf, typename OutputOf<kMode>::Type* d_min_max,
                cudaStream_t stream, cudaEvent_t* pass_events = nullptr)
{
  const int64_t count = nx * ny * nz;
  StreamScratch<uint32_t> scratch;
  VGT_CUDA_TRY(scratch.Allocate(count, stream), "SDF scratch allocation");
  uint32_t* d_front = reinterpret_cast<uint32_t*>(d_sdf);
  // After the local passes the packed field must sit in the scratch (the final pass writes d_sdf).
  if (pass_events != nullptr)
  {
    cudaEventRecord(pass_events[0], stream);
  }
  int status = VGT_B200_OK;
  if (ny <= 1)
  {
    status = LaunchScan<In>(d_in, scratch.get(), nx * ny, static_cast<int32_t>(nz),
                            unknown_is_filled, stream);
    if (pass_events != nullptr)
    {
      cudaEventRecord(pass_events[1], stream);
    }
  }
  else
  {
    status = LaunchScan<In>(d_in, d_front, nx * ny, static_cast<int32_t>(nz), unknown_is_filled,
                            stream);
    if (pass_events != nullptr)
    {
      cudaEventRecord(pass_events[1], stream);
    }
    if (status == VGT_B200_OK)
    {
      status = LaunchEnvelope<kEmitPacked>(d_front, scratch.get(), FamilyAlongY(nx, ny, nz),
                                           Square(nz - 1), FinalizeParams{}, nullptr, stream);
    }
  }
  if (pass_events != nullptr)
  {
    cudaEventRecord(pass_events[2], stream);
  }
  if (status != VGT_B200_OK)
  {
    return status;
  }
  status = RunFinalPass<kMode>(scratch.get(), nx, ny, nz, 0, ny, resolution, add_virtual_border,
                               d_sdf, d_min_max, stream);
  if (pass_events != nullptr)
  {
    cudaEventRecord(pass_events[3], stream);
  }
  return status;
}

// Grids above this size go through the pipelined host path (copies overlapped with the passes).
constexpr int64_t kPipelineMinVoxels = int64_t{1} << 24;
constexpr int kPipelineChunks = 8;

// x envelope + finalize on the column range [y0 * nz, y1 * nz) of a FULL grid [nx, ny, nz] (line
// stride ny * nz): the y-chunked final pass of the pipelined host path. Keys are reset / decoded
// by the caller. d_packed is destroyed in that range.
template <int kMode>
int RunFinalPassColumns(uint32_t* d_packed, int64_t nx, int64_t ny, int64_t nz, int64_t y0,
                        int64_t y1, double resolution, int add_virtual_border,
                        typename OutputOf<kMode>::Type* d_out,
                        typename OutputOf<kMode>::Key* d_keys,
                        const MagnitudeTable<typename OutputOf<kMode>::Type>& magnitudes,
                        cudaStream_t stream)
{
  FinalizeParams finalize{};
  magnitudes.Attach(finalize);
  finalize.resolution = resolution;
  finalize.add_virtual_border = add_virtual_border;
  finalize.nx_total = static_cast<int32_t>(nx);
  finalize.ny_total = static_cast<int32_t>(ny);
  finalize.nz_total = static_cast<int32_t>(nz);
  finalize.y_offset = static_cast<int32_t>(y0);
  finalize.nz = static_cast<int32_t>(nz);
  const LineFamily family{1, 0, (y1 - y0) * nz, ny * nz, static_cast<int32_t>(nx)};
  return LaunchEnvelope<kMode>(d_packed + y0 * nz, d_out + y0 * nz, family,
                               Square(nz - 1) + Square(ny - 1), finalize, d_keys, stream);
}

// Host-pointer entry for large grids: the input arrives in x-slabs, and the z and y passes of a
// slab (independent per x) run while the next slab is still on the bus; the x pass + finalize
// runs in y-slabs, each copied back (a strided 2-D copy) while the next one is computed. PCIe
// stays busy from the first byte in to the last byte out; only one slab of compute is exposed
// at either end.
template <typename In, int kMode>
int SdfFromHostPipelined(const In* h_in, int64_t nx, int64_t ny, int64_t nz, double resolution,
                         int unknown_is_filled, int add_virtual_border,
                         typename OutputOf<kMode>::Type* h_out,
                         typename OutputOf<kMode>::Type* out_min,
                         typename OutputOf<kMode>::Type* out_max)
{
  using Out = typename OutputOf<kMode>::Type;
  using Key = typename OutputOf<kMode>::Key;
  const int64_t count = nx * ny * nz;
  const int64_t plane = ny * nz;
  StreamGuard compute, copy_in, copy_out;
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&compute.stream, cudaStreamNonBlocking), "stream");
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&copy_in.stream, cudaStreamNonBlocking), "stream");
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&copy_out.stream, cudaStreamNonBlocking), "stream");
  StreamScratch<In> d_in;
  StreamScratch<Out> d_out;
  StreamScratch<uint32_t> scratch;
  StreamScratch<Out> d_min_max;
  StreamScratch<Key> keys;
  VGT_CUDA_TRY(d_in.Allocate(count, compute.stream), "input grid allocation");
  VGT_CUDA_TRY(d_out.Allocate(count, compute.stream), "SDF allocation");
  VGT_CUDA_TRY(scratch.Allocate(count, compute.stream), "SDF scratch allocation");
  VGT_CUDA_TRY(d_min_max.Allocate(2, compute.stream), "min/max allocation");
  VGT_CUDA_TRY(keys.Allocate(2, compute.stream), "min/max scratch");
  ResetMinMaxKeysKernel<Key><<<1, 1, 0, compute.stream>>>(keys.get()); NoteKernelLaunch();
  EventGuard allocated;
  VGT_CUDA_TRY(cudaEventCreateWithFlags(&allocated.event, cudaEventDisableTiming), "event");
  VGT_CUDA_TRY(cudaEventRecord(allocated.event, compute.stream), "event record");
  VGT_CUDA_TRY(cudaStreamWaitEvent(copy_in.stream, allocated.event, 0), "stream wait");
  VGT_CUDA_TRY(cudaStreamWaitEvent(copy_out.stream, allocated.event, 0), "stream wait");

  uint32_t* const d_front = reinterpret_cast<uint32_t*>(d_out.get());
  // pageable caller buffers go through pinned slots filled / drained by several host threads
  StagedTransfer transfer;
  // Declared after the buffers and the staging object, so it runs first on every exit path
  // (early error returns included): nothing of this call is still queued when the pinned slots
  // go back to the process-wide cache and the scratch to the pool.
  struct DrainOnExit
  {
    cudaStream_t streams[3];
    ~DrainOnExit()
    {
      for (cudaStream_t stream : streams)
      {
        cudaStreamSynchronize(stream);
      }
    }
  } drain{{copy_in.stream, compute.stream, copy_out.stream}};
  const int in_chunks = static_cast<int>(nx < kPipelineChunks ? nx : kPipelineChunks);
  EventGuard arrived[kPipelineChunks];
  int status = VGT_B200_OK;
  for (int c = 0; c < in_chunks && status == VGT_B200_OK; c++)
  {
    const int64_t x0 = nx * c / in_chunks;
    const int64_t x1 = nx * (c + 1) / in_chunks;
    {
      const size_t slab_bytes = sizeof(In) * static_cast<size_t>((x1 - x0) * plane);
      VGT_CUDA_TRY(transfer.ToDevice(reinterpret_cast<char*>(d_in.get() + x0 * plane), slab_bytes,
                                     reinterpret_cast<const char*>(h_in + x0 * plane), slab_bytes,
                                     slab_bytes, 1, copy_in.stream),
                   "copy grid slab to device");
    }
    VGT_CUDA_TRY(cudaEventCreateWithFlags(&arrived[c].event, cudaEventDisableTiming), "event");
    VGT_CUDA_TRY(cudaEventRecord(arrived[c].event, copy_in.stream), "event record");
    VGT_CUDA_TRY(cudaStreamWaitEvent(compute.stream, arrived[c].event, 0), "stream wait");
    // z scan into the front buffer, y envelope into the scratch (or z scan straight into the
    // scratch when there is no y axis): after this the packed field of the slab is in `scratch`.
    if (ny <= 1)
    {
      status = LaunchScan<In>(d_in.get() + x0 * plane, scratch.get() + x0 * plane,
                              (x1 - x0) * ny, static_cast<int32_t>(nz), unknown_is_filled,
                              compute.stream);
    }
    else
    {
      status = LaunchScan<In>(d_in.get() + x0 * plane, d_front + x0 * plane, (x1 - x0) * ny,
                              static_cast<int32_t>(nz), unknown_is_filled, compute.stream);
      if (status == VGT_B200_OK)
      {
        status = LaunchEnvelope<kEmitPacked>(d_front + x0 * plane, scratch.get() + x0 * plane,
                                             FamilyAlongY(x1 - x0, ny, nz), Square(nz - 1),
                                             FinalizeParams{}, nullptr, compute.stream);
      }
    }
  }
  MagnitudeTable<Out> magnitudes;
  if (status == VGT_B200_OK)
  {
    status = magnitudes.Build(nx, ny, nz, resolution, compute.stream);
  }
  const int out_chunks = static_cast<int>(ny < kPipelineChunks ? ny : kPipelineChunks);
  EventGuard finished[kPipelineChunks];
  // every y-slab of the final pass is enqueued first (the compute stream never waits for the
  // host), then the slabs are copied out in order, each as soon as its pass has finished
  for (int c = 0; c < out_chunks && status == VGT_B200_OK; c++)
  {
    const int64_t y0 = ny * c / out_chunks;
    const int64_t y1 = ny * (c + 1) / out_chunks;
    status = RunFinalPassColumns<kMode>(scratch.get(), nx, ny, nz, y0, y1, resolution,
                                        add_virtual_border, d_out.get(), keys.get(), magnitudes,
                                        compute.stream);
    if (status != VGT_B200_OK)
    {
      break;
    }
    VGT_CUDA_TRY(cudaEventCreateWithFlags(&finished[c].event, cudaEventDisableTiming), "event");
    VGT_CUDA_TRY(cudaEventRecord(finished[c].event, compute.stream), "event record");
  }
  Out min_max[2];
  if (status == VGT_B200_OK)
  {
    DecodeMinMaxKernel<Out, Key><<<1, 1, 0, compute.stream>>>(keys.get(), d_min_max.get()); NoteKernelLaunch();
  }
  for (int c = 0; c < out_chunks && status == VGT_B200_OK; c++)
  {
    const int64_t y0 = ny * c / out_chunks;
    const int64_t y1 = ny * (c + 1) / out_chunks;
    VGT_CUDA_TRY(cudaStreamWaitEvent(copy_out.stream, finished[c].event, 0), "stream wait");
    // rows = x planes, one row = the slab's (y1 - y0) * nz values (a strided 2-D copy)
    VGT_CUDA_TRY(transfer.ToHost(reinterpret_cast<char*>(h_out + y0 * nz), sizeof(Out) * plane,
                                 reinterpret_cast<const char*>(d_out.get() + y0 * nz),
                                 sizeof(Out) * plane, sizeof(Out) * (y1 - y0) * nz,
                                 static_cast<size_t>(nx), copy_out.stream),
                 "copy SDF slab to host");
  }
  if (status == VGT_B200_OK)
  {
    // (after the copy-out loop: a device-to-host copy into pageable memory blocks the host
    // until the compute stream has drained, which would serialise the slab copies behind it)
    cudaMemcpyAsync(min_max, d_min_max.get(), sizeof(Out) * 2, cudaMemcpyDeviceToHost,
                    compute.stream);
  }
  const cudaError_t sync_in = cudaStreamSynchronize(copy_in.stream);
  const cudaError_t sync_compute = cudaStreamSynchronize(compute.stream);
  const cudaError_t sync_out = cudaStreamSynchronize(copy_out.stream);
  if (status != VGT_B200_OK)
  {
    return status;
  }
  VGT_CUDA_TRY(sync_in, "copy grid to device");
  VGT_CUDA_TRY(sync_compute, "SDF generation");
  VGT_CUDA_TRY(sync_out, "copy SDF to host");
  if (out_min != nullptr)
  {
    *out_min = min_max[0];
  }
  if (out_max != nullptr)
  {
    *out_max = min_max[1];
  }
  return VGT_B200_OK;
}

// Host-pointer entry: allocate, copy in, run, copy out, synchronise.
template <typename In, int kMode>
int SdfFromHost(const In* h_in, int64_t nx, int64_t ny, int64_t nz, double resolution,
                int unknown_is_filled, int add_virtual_border, int device,
                typename OutputOf<kMode>::Type* h_out, typename OutputOf<kMode>::Type* out_min,
                typename OutputOf<kMode>::Type* out_max)
{
  using Out = typename OutputOf<kMode>::Type;
  const int check = CheckSdfArguments(h_in, h_out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  const int64_t count = nx * ny * nz;
  if (count >= kPipelineMinVoxels && nx > 1)
  {
    return SdfFromHostPipelined<In, kMode>(h_in, nx, ny, nz, resolution, unknown_is_filled,
                                           add_virtual_border, h_out, out_min, out_max);
  }
  StreamGuard guard;
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&guard.stream, cudaStreamNonBlocking),
               "cudaStreamCreate");
  cudaStream_t stream = guard.stream;
  StreamScratch<In> d_in;
  StreamScratch<Out> d_out;
  StreamScratch<Out> d_min_max;
  VGT_CUDA_TRY(d_in.Allocate(count, stream), "input grid allocation");
  VGT_CUDA_TRY(d_out.Allocate(count, stream), "SDF allocation");
  VGT_CUDA_TRY(d_min_max.Allocate(2, stream), "min/max allocation");
  VGT_CUDA_TRY(cudaMemcpyAsync(d_in.get(), h_in, sizeof(In) * count, cudaMemcpyHostToDevice,
                               stream),
               "copy grid to device");
  const int status =
      SdfOnDevice<In, kMode>(d_in.get(), nx, ny, nz, resolution, unknown_is_filled,
                             add_virtual_border, d_out.get(), d_min_max.get(), stream);
  if (status != VGT_B200_OK)
  {
    cudaStreamSynchronize(stream);
    return status;
  }
  Out min_max[2];
  VGT_CUDA_TRY(cudaMemcpyAsync(h_out, d_out.get(), sizeof(Out) * count, cudaMemcpyDeviceToHost,
                               stream),
               "copy SDF to host");
  VGT_CUDA_TRY(cudaMemcpyAsync(min_max, d_min_max.get(), sizeof(Out) * 2, cudaMemcpyDeviceToHost,
                               stream),
               "copy min/max to host");
  VGT_CUDA_TRY(cudaStreamSynchronize(stream), "SDF generation");
  if (out_min != nullptr)
  {
    *out_min = min_max[0];
  }
  if (out_max != nullptr)
  {
    *out_max = min_max[1];
  }
  return VGT_B200_OK;
}
// ------------------------------------------------------------------------------------------------
// Other map types: cells { float occupancy; uint32 object_id; ... } (edt_cells.cuh)
// ------------------------------------------------------------------------------------------------
int CheckCellArguments(const void* cells, int cell_bytes, const void* out, int64_t nx, int64_t ny,
                       int64_t nz, double resolution, const uint32_t* object_ids,
                       int64_t num_object_ids)
{
  const int check = CheckSdfArguments(cells, out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (cell_bytes != 8 && cell_bytes != 16)
  {
    return FailInvalid("cell size must be 8 or 16 bytes, got %d", cell_bytes);
  }
  if (num_object_ids < 0 || num_object_ids > 0x7fffffffLL
      || (num_object_ids > 0 && object_ids == nullptr))
  {
    return FailInvalid("invalid object id list");
  }
  return VGT_B200_OK;
}

// Device-resident cells -> SDF of the voxels the rule marks filled.
template <int kMode>
int SdfFromCellsOnDevice(const uint32_t* d_cells, int cell_words, int64_t nx, int64_t ny,
                         int64_t nz, double resolution, int unknown_is_filled,
                         int add_virtual_border, int object_rule, const uint32_t* d_sorted_ids,
                         int num_ids, typename OutputOf<kMode>::Type* d_sdf,
                         typename OutputOf<kMode>::Type* d_min_max, cudaStream_t stream)
{
  const int64_t count = nx * ny * nz;
  StreamScratch<uint8_t> mask;
  VGT_CUDA_TRY(mask.Allocate(count, stream), "filled mask allocation");
  const int threads = 256;
  CellsToMaskKernel<<<static_cast<unsigned>((count + threads - 1) / threads), threads, 0,
                      stream>>>(d_cells, cell_words, count, unknown_is_filled, object_rule,
                                d_sorted_ids, num_ids, mask.get()); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "CellsToMaskKernel launch");
  return SdfOnDevice<uint8_t, kMode>(mask.get(), nx, ny, nz, resolution, 0, add_virtual_border,
                                     d_sdf, d_min_max, stream);
}

std::vector<uint32_t> SortedDistinct(const uint32_t* object_ids, int64_t num_object_ids)
{
  std::vector<uint32_t> sorted(object_ids, object_ids + num_object_ids);
  std::sort(sorted.begin(), sorted.end());
  sorted.erase(std::unique(sorted.begin(), sorted.end()), sorted.end());
  return sorted;
}

// The id list of CellsToMaskKernel on the device (nothing is allocated for an empty list). The
// copy from pageable memory has read `sorted` when cudaMemcpyAsync returns.
int UploadIds(const std::vector<uint32_t>& sorted, StreamScratch<uint32_t>& ids,
              cudaStream_t stream)
{
  if (!sorted.empty())
  {
    VGT_CUDA_TRY(ids.Allocate(static_cast<int64_t>(sorted.size()), stream), "id allocation");
    VGT_CUDA_TRY(cudaMemcpyAsync(ids.get(), sorted.data(), sizeof(uint32_t) * sorted.size(),
                                 cudaMemcpyHostToDevice, stream),
                 "copy object ids to device");
  }
  return VGT_B200_OK;
}

// Cells and (sorted) object ids uploaded once for one or several SDFs.
struct CellUpload
{
  StreamScratch<uint32_t> cells;
  StreamScratch<uint32_t> ids;
  std::vector<uint32_t> sorted;
  int Upload(const void* h_cells, int cell_bytes, int64_t count, const uint32_t* object_ids,
             int64_t num_object_ids, cudaStream_t stream)
  {
    VGT_CUDA_TRY(cells.Allocate(count * (cell_bytes / 4), stream), "cell array allocation");
    {
      // (pageable std::vector storage goes through the pinned staging ring)
      StagedTransfer transfer;
      const size_t bytes = static_cast<size_t>(count) * cell_bytes;
      VGT_CUDA_TRY(transfer.ToDevice(reinterpret_cast<char*>(cells.get()), bytes,
                                     static_cast<const char*>(h_cells), bytes, bytes, 1, stream),
                   "copy cells to device");
      // the slots go back to the cache when `transfer` dies: their DMA must have finished
      VGT_CUDA_TRY(cudaStreamSynchronize(stream), "copy cells to device");
    }
    sorted = SortedDistinct(object_ids, num_object_ids);
    return UploadIds(sorted, ids, stream);
  }
};

// num_sdfs == 1: one SDF of the cells whose object id is in object_ids (all objects when the
// list is empty). per_object: one SDF per listed object id (MakeSeparateObjectSDFs), results
// back to back in h_out.
template <int kMode>
int SdfFromCellsHost(const void* h_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                     double resolution, int unknown_is_filled, int add_virtual_border,
                     const uint32_t* object_ids, int64_t num_object_ids, bool per_object,
                     int device, typename OutputOf<kMode>::Type* h_out,
                     typename OutputOf<kMode>::Type* out_min,
                     typename OutputOf<kMode>::Type* out_max)
{
  using Out = typename OutputOf<kMode>::Type;
  const int check = CheckCellArguments(h_cells, cell_bytes, h_out, nx, ny, nz, resolution,
                                       object_ids, num_object_ids);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  const int64_t count = nx * ny * nz;
  StreamGuard guard;
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&guard.stream, cudaStreamNonBlocking),
               "cudaStreamCreate");
  cudaStream_t stream = guard.stream;
  CellUpload upload;
  const int uploaded = upload.Upload(h_cells, cell_bytes, count, object_ids,
                                     per_object ? 0 : num_object_ids, stream);
  if (uploaded != VGT_B200_OK)
  {
    return uploaded;
  }
  const int64_t num_sdfs = per_object ? num_object_ids : 1;
  // Two result buffers and a copy stream: the SDF of object k + 1 is computed while object k
  // travels to the host (through the pinned staging ring when the caller's buffer is pageable).
  StreamGuard copy;
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&copy.stream, cudaStreamNonBlocking), "cudaStreamCreate");
  StreamScratch<Out> d_out[2];
  StreamScratch<Out> d_min_max;
  StreamScratch<uint32_t> d_one_id;
  VGT_CUDA_TRY(d_out[0].Allocate(count, stream), "SDF allocation");
  if (num_sdfs > 1)
  {
    VGT_CUDA_TRY(d_out[1].Allocate(count, stream), "SDF allocation");
  }
  VGT_CUDA_TRY(d_min_max.Allocate(2 * std::max<int64_t>(num_sdfs, 1), stream), "min/max");
  if (per_object && num_sdfs > 0)
  {
    VGT_CUDA_TRY(d_one_id.Allocate(num_sdfs, stream), "id allocation");
    VGT_CUDA_TRY(cudaMemcpyAsync(d_one_id.get(), object_ids, sizeof(uint32_t) * num_sdfs,
                                 cudaMemcpyHostToDevice, stream),
                 "copy object ids to device");
  }
  StagedTransfer transfer;
  EventGuard computed[2];
  for (auto& guard_event : computed)
  {
    VGT_CUDA_TRY(cudaEventCreateWithFlags(&guard_event.event, cudaEventDisableTiming), "event");
  }
  // (runs first on every exit path: nothing is still queued when the buffers are released)
  struct DrainOnExit
  {
    cudaStream_t a;
    cudaStream_t b;
    ~DrainOnExit()
    {
      cudaStreamSynchronize(a);
      cudaStreamSynchronize(b);
    }
  } drain{stream, copy.stream};
  const auto enqueue = [&](int64_t k) -> int
  {
    Out* const target = d_out[k & 1].get();
    int status;
    if (per_object)
    {
      status = SdfFromCellsOnDevice<kMode>(upload.cells.get(), cell_bytes / 4, nx, ny, nz,
                                           resolution, unknown_is_filled, add_virtual_border,
                                           kListedObjects, d_one_id.get() + k, 1, target,
                                           d_min_max.get() + 2 * k, stream);
    }
    else
    {
      const int num_ids = static_cast<int>(upload.sorted.size());
      status = SdfFromCellsOnDevice<kMode>(upload.cells.get(), cell_bytes / 4, nx, ny, nz,
                                           resolution, unknown_is_filled, add_virtual_border,
                                           num_ids > 0 ? kListedObjects : kAnyObject,
                                           upload.ids.get(), num_ids, target, d_min_max.get(),
                                           stream);
    }
    if (status != VGT_B200_OK)
    {
      return status;
    }
    VGT_CUDA_TRY(cudaEventRecord(computed[k & 1].event, stream), "event record");
    return VGT_B200_OK;
  };
  std::vector<Out> min_max(static_cast<size_t>(2 * std::max<int64_t>(num_sdfs, 1)));
  if (num_sdfs > 0)
  {
    const int status = enqueue(0);
    if (status != VGT_B200_OK)
    {
      return status;
    }
  }
  for (int64_t k = 0; k < num_sdfs; k++)
  {
    if (k + 1 < num_sdfs)
    {
      // (buffer (k + 1) & 1 was drained by the blocking copy of object k - 1)
      const int status = enqueue(k + 1);
      if (status != VGT_B200_OK)
      {
        return status;
      }
    }
    VGT_CUDA_TRY(cudaStreamWaitEvent(copy.stream, computed[k & 1].event, 0), "stream wait");
    const size_t bytes = sizeof(Out) * static_cast<size_t>(count);
    VGT_CUDA_TRY(transfer.ToHost(reinterpret_cast<char*>(h_out + k * count), bytes,
                                 reinterpret_cast<const char*>(d_out[k & 1].get()), bytes, bytes,
                                 1, copy.stream),
                 "copy SDF to host");
    VGT_CUDA_TRY(cudaStreamSynchronize(copy.stream), "copy SDF to host");
  }
  if (num_sdfs > 0)
  {
    VGT_CUDA_TRY(cudaMemcpyAsync(min_max.data(), d_min_max.get(), sizeof(Out) * 2 * num_sdfs,
                                 cudaMemcpyDeviceToHost, stream),
                 "copy min/max to host");
  }
  VGT_CUDA_TRY(cudaStreamSynchronize(stream), "SDF generation from cells");
  for (int64_t k = 0; k < num_sdfs; k++)
  {
    if (out_min != nullptr)
    {
      out_min[k] = min_max[2 * k];
    }
    if (out_max != nullptr)
    {
      out_max[k] = min_max[2 * k + 1];
    }
  }
  return VGT_B200_OK;
}

// ExtractFreeAndNamedObjectsSignedDistanceField (tagged_object_occupancy_map.hpp:293-378) on
// device-resident cells: the SDF of every filled cell into d_sdf, the SDF of the filled cells of
// named objects (id > 0) into a scratch, merged into d_sdf. d_min_max may be null.
template <int kMode>
int SdfFreeAndNamedOnDevice(const uint32_t* d_cells, int cell_words, int64_t nx, int64_t ny,
                            int64_t nz, double resolution, int unknown_is_filled,
                            int add_virtual_border, typename OutputOf<kMode>::Type* d_sdf,
                            typename OutputOf<kMode>::Type* d_min_max, cudaStream_t stream)
{
  using Out = typename OutputOf<kMode>::Type;
  using Key = typename OutputOf<kMode>::Key;
  const int64_t count = nx * ny * nz;
  StreamScratch<Out> d_named;
  StreamScratch<Key> keys;
  VGT_CUDA_TRY(d_named.Allocate(count, stream), "SDF allocation");
  if (d_min_max != nullptr)
  {
    VGT_CUDA_TRY(keys.Allocate(2, stream), "min/max scratch");
  }
  int status = SdfFromCellsOnDevice<kMode>(d_cells, cell_words, nx, ny, nz, resolution,
                                           unknown_is_filled, add_virtual_border, kAnyObject,
                                           nullptr, 0, d_sdf, nullptr, stream);
  if (status == VGT_B200_OK)
  {
    status = SdfFromCellsOnDevice<kMode>(d_cells, cell_words, nx, ny, nz, resolution,
                                         unknown_is_filled, add_virtual_border, kNamedObjects,
                                         nullptr, 0, d_named.get(), nullptr, stream);
  }
  if (status != VGT_B200_OK)
  {
    return status;
  }
  if (d_min_max != nullptr)
  {
    ResetMinMaxKeysKernel<Key><<<1, 1, 0, stream>>>(keys.get()); NoteKernelLaunch();
  }
  const int threads = 256;
  const int64_t merge_blocks =
      std::min<int64_t>((count + threads - 1) / threads, MultiprocessorCount() * 16);
  MergeFreeAndNamedKernel<Out, Key><<<static_cast<unsigned>(merge_blocks), threads, 0, stream>>>(
          d_sdf, d_named.get(), count, d_sdf, keys.get()); NoteKernelLaunch();
  if (d_min_max != nullptr)
  {
    DecodeMinMaxKernel<Out, Key><<<1, 1, 0, stream>>>(keys.get(), d_min_max); NoteKernelLaunch();
  }
  VGT_CUDA_TRY(cudaGetLastError(), "MergeFreeAndNamedKernel launch");
  return VGT_B200_OK;
}

// The same on host cells, with the upload and the copy-out.
template <int kMode>
int SdfFreeAndNamedHost(const void* h_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                        double resolution, int unknown_is_filled, int add_virtual_border,
                        int device, typename OutputOf<kMode>::Type* h_out,
                        typename OutputOf<kMode>::Type* out_min,
                        typename OutputOf<kMode>::Type* out_max)
{
  using Out = typename OutputOf<kMode>::Type;
  const int check = CheckCellArguments(h_cells, cell_bytes, h_out, nx, ny, nz, resolution,
                                       nullptr, 0);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  const int64_t count = nx * ny * nz;
  StreamGuard guard;
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&guard.stream, cudaStreamNonBlocking),
               "cudaStreamCreate");
  cudaStream_t stream = guard.stream;
  CellUpload upload;
  const int uploaded = upload.Upload(h_cells, cell_bytes, count, nullptr, 0, stream);
  if (uploaded != VGT_B200_OK)
  {
    return uploaded;
  }
  StreamScratch<Out> d_free;
  StreamScratch<Out> d_min_max;
  VGT_CUDA_TRY(d_free.Allocate(count, stream), "SDF allocation");
  VGT_CUDA_TRY(d_min_max.Allocate(2, stream), "min/max allocation");
  const int status = SdfFreeAndNamedOnDevice<kMode>(upload.cells.get(), cell_bytes / 4, nx, ny,
                                                    nz, resolution, unknown_is_filled,
                                                    add_virtual_border, d_free.get(),
                                                    d_min_max.get(), stream);
  if (status != VGT_B200_OK)
  {
    cudaStreamSynchronize(stream);
    return status;
  }
  Out min_max[2];
  VGT_CUDA_TRY(cudaMemcpyAsync(h_out, d_free.get(), sizeof(Out) * count, cudaMemcpyDeviceToHost,
                               stream),
               "copy SDF to host");
  VGT_CUDA_TRY(cudaMemcpyAsync(min_max, d_min_max.get(), sizeof(Out) * 2, cudaMemcpyDeviceToHost,
                               stream),
               "copy min/max to host");
  VGT_CUDA_TRY(cudaStreamSynchronize(stream), "free-and-named SDF generation");
  if (out_min != nullptr)
  {
    *out_min = min_max[0];
  }
  if (out_max != nullptr)
  {
    *out_max = min_max[1];
  }
  return VGT_B200_OK;
}

// The cell entries on device pointers (vgt_b200_sdf_*_dev): asynchronous on the caller's stream.
// Every argument is checked before the first device call: the host entries' checks, and the
// alignment the kernels read and write with.
template <int kMode>
int CheckDeviceCellArguments(const void* d_cells, int cell_bytes, int64_t nx, int64_t ny,
                             int64_t nz, double resolution, const uint32_t* object_ids,
                             int64_t num_object_ids, const typename OutputOf<kMode>::Type* d_sdf,
                             const typename OutputOf<kMode>::Type* d_min_max)
{
  using Out = typename OutputOf<kMode>::Type;
  const int check = CheckCellArguments(d_cells, cell_bytes, d_sdf, nx, ny, nz, resolution,
                                       object_ids, num_object_ids);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (reinterpret_cast<uintptr_t>(d_cells) % 4 != 0)
  {
    return FailInvalid("cell array must be 4-byte aligned");
  }
  if (reinterpret_cast<uintptr_t>(d_sdf) % sizeof(Out) != 0
      || reinterpret_cast<uintptr_t>(d_min_max) % sizeof(Out) != 0)
  {
    return FailInvalid("SDF and min/max arrays must be aligned to their scalar type");
  }
  return VGT_B200_OK;
}

template <int kMode>
int SdfFromCellsDev(const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                    double resolution, int unknown_is_filled, int add_virtual_border,
                    const uint32_t* object_ids, int64_t num_object_ids, int device,
                    typename OutputOf<kMode>::Type* d_sdf,
                    typename OutputOf<kMode>::Type* d_min_max, cudaStream_t stream)
{
  const int check = CheckDeviceCellArguments<kMode>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                                    object_ids, num_object_ids, d_sdf, d_min_max);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  const std::vector<uint32_t> sorted = SortedDistinct(object_ids, num_object_ids);
  StreamScratch<uint32_t> ids;
  const int uploaded = UploadIds(sorted, ids, stream);
  if (uploaded != VGT_B200_OK)
  {
    return uploaded;
  }
  const int num_ids = static_cast<int>(sorted.size());
  return SdfFromCellsOnDevice<kMode>(static_cast<const uint32_t*>(d_cells), cell_bytes / 4, nx,
                                     ny, nz, resolution, unknown_is_filled, add_virtual_border,
                                     num_ids > 0 ? kListedObjects : kAnyObject, ids.get(),
                                     num_ids, d_sdf, d_min_max, stream);
}

// MakeSeparateObjectSDFs on device cells: SDF k of the k-th listed id at d_sdf + k * V, its
// min/max at d_min_max + 2 k. The distinct ids go in groups of kSlotGroupSize; each group's slot
// map is built with one read of the cells and serves the SDFs of every listed id in the group.
template <int kMode>
int SdfPerObjectDev(const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                    double resolution, int unknown_is_filled, int add_virtual_border,
                    const uint32_t* object_ids, int64_t num_object_ids, int device,
                    typename OutputOf<kMode>::Type* d_sdf,
                    typename OutputOf<kMode>::Type* d_min_max, cudaStream_t stream)
{
  using Out = typename OutputOf<kMode>::Type;
  const int check = CheckDeviceCellArguments<kMode>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                                    object_ids, num_object_ids, d_sdf, d_min_max);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  const int64_t count = nx * ny * nz;
  if (num_object_ids > 0
      && count * static_cast<int64_t>(sizeof(Out)) > INT64_MAX / num_object_ids)
  {
    return FailInvalid("%lld SDFs of %lld voxels overflow a 64-bit byte count",
                       static_cast<long long>(num_object_ids), static_cast<long long>(count));
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  if (num_object_ids == 0)
  {
    return VGT_B200_OK;
  }
  KeepPoolMemory(device);
  const std::vector<uint32_t> sorted = SortedDistinct(object_ids, num_object_ids);
  std::vector<int64_t> position(static_cast<size_t>(num_object_ids));
  for (int64_t k = 0; k < num_object_ids; k++)
  {
    position[k] = std::lower_bound(sorted.begin(), sorted.end(), object_ids[k]) - sorted.begin();
  }
  StreamScratch<uint8_t> slots;
  VGT_CUDA_TRY(slots.Allocate(count, stream), "object slot map allocation");
  const ObjectSlot* const d_slots = reinterpret_cast<const ObjectSlot*>(slots.get());
  const int threads = 256;
  const int64_t blocks = std::min<int64_t>((count + threads * 4 - 1) / (threads * 4),
                                           MultiprocessorCount() * 8);
  for (int64_t first = 0; first < static_cast<int64_t>(sorted.size()); first += kSlotGroupSize)
  {
    SlotGroup group{};
    group.count = static_cast<int>(
        std::min<int64_t>(kSlotGroupSize, static_cast<int64_t>(sorted.size()) - first));
    std::copy(sorted.begin() + first, sorted.begin() + first + group.count, group.ids);
    CellsToObjectSlotsKernel<<<static_cast<unsigned>(blocks), threads, 0, stream>>>(
        static_cast<const uint32_t*>(d_cells), cell_bytes / 4, count, unknown_is_filled, group,
        slots.get()); NoteKernelLaunch();
    VGT_CUDA_TRY(cudaGetLastError(), "CellsToObjectSlotsKernel launch");
    for (int64_t k = 0; k < num_object_ids; k++)
    {
      if (position[k] < first || position[k] >= first + group.count)
      {
        continue;
      }
      const int key = static_cast<int>(position[k] - first) + 1;
      const int status = SdfOnDevice<ObjectSlot, kMode>(
          d_slots, nx, ny, nz, resolution, key, add_virtual_border, d_sdf + k * count,
          d_min_max == nullptr ? nullptr : d_min_max + 2 * k, stream);
      if (status != VGT_B200_OK)
      {
        return status;
      }
    }
  }
  return VGT_B200_OK;
}

template <int kMode>
int SdfFreeAndNamedDev(const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz,
                       double resolution, int unknown_is_filled, int add_virtual_border,
                       int device, typename OutputOf<kMode>::Type* d_sdf,
                       typename OutputOf<kMode>::Type* d_min_max, cudaStream_t stream)
{
  const int check = CheckDeviceCellArguments<kMode>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                                    nullptr, 0, d_sdf, d_min_max);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  return SdfFreeAndNamedOnDevice<kMode>(static_cast<const uint32_t*>(d_cells), cell_bytes / 4, nx,
                                        ny, nz, resolution, unknown_is_filled, add_virtual_border,
                                        d_sdf, d_min_max, stream);
}
// ------------------------------------------------------------------------------------------------
// One process, several devices: the slab-sharded path of voxelized_geometry_tools_b200/sharded.py
// behind one C call, so that a C++ caller of the SDF members can use every GPU of the box, and a
// map that one device cannot hold gets its SDF. One host thread per device runs that device's
// share: upload of its x-slab, z scan + y pass with the exchange fused in (peer stores into the
// other devices' receive buffers: cudaMalloc memory with peer access enabled), a barrier between
// the threads once every stream has drained, x pass + finalize on its y-slab, strided copy of the
// y-slab into its place in the caller's grid. A call runs one or more such rounds on the same
// resident input slab (free-and-named: two; the per-object batch: one per listed id).
// ------------------------------------------------------------------------------------------------

// The grid of a multi-device call and its cut: x-slab g of the input and y-slab g of the result
// belong to devices[g].
struct MultiGrid
{
  int64_t nx, ny, nz;
  double resolution;
  int add_virtual_border;
  int num_devices;
  int64_t Plane() const { return ny * nz; }
};

// What the per-slab steps of one device see.
struct SlabPart
{
  int index;
  int64_t x0, x1, y0, y1;
  cudaStream_t stream;
  StagedTransfer* transfer;
  uint32_t* scratch;            // 4 bytes per voxel of the x-slab, the z scan's output
  const uint64_t* peer_bases;   // every device's receive buffer
  int64_t Voxels(const MultiGrid& grid) const { return (x1 - x0) * grid.Plane(); }
};

// z scan of the part's input slab, then the y pass, whose output goes straight into every
// device's receive buffer.
template <typename In>
int ExchangeLocalPasses(const In* d_slab, int unknown_is_filled, const MultiGrid& grid,
                        const SlabPart& part)
{
  return RunLocalPasses<In>(d_slab, part.x1 - part.x0, grid.ny, grid.nz, unknown_is_filled,
                            part.scratch, part.scratch, part.stream, grid.num_devices,
                            part.peer_bases, part.x0, part.index);
}

// y-slab [nx][rows][nz] -> rows [y0, y1) of the caller's [nx][ny][nz] grid (a strided 2-D
// copy), and the slab's min/max into h_min_max[2]. Both land when the stream has drained.
template <typename Out>
int CopySlabToHost(const Out* d_slab, const Out* d_min_max, const MultiGrid& grid,
                   const SlabPart& part, Out* h_grid, Out* h_min_max)
{
  const int64_t rows = part.y1 - part.y0;
  VGT_CUDA_TRY(part.transfer->ToHost(reinterpret_cast<char*>(h_grid + part.y0 * grid.nz),
                                     sizeof(Out) * static_cast<size_t>(grid.Plane()),
                                     reinterpret_cast<const char*>(d_slab),
                                     sizeof(Out) * static_cast<size_t>(rows * grid.nz),
                                     sizeof(Out) * static_cast<size_t>(rows * grid.nz),
                                     static_cast<size_t>(grid.nx), part.stream),
               "copy SDF slab to host");
  VGT_CUDA_TRY(cudaMemcpyAsync(h_min_max, d_min_max, sizeof(Out) * 2, cudaMemcpyDeviceToHost,
                               part.stream),
               "copy min/max to host");
  return VGT_B200_OK;
}

// extrema: [result][device][min, max] -> out_min[result], out_max[result] (either may be null).
template <typename Out>
void CombineExtrema(const std::vector<Out>& extrema, int num_devices, int64_t results,
                    Out* out_min, Out* out_max)
{
  for (int64_t k = 0; k < results; k++)
  {
    const Out* row = extrema.data() + 2 * k * num_devices;
    Out low = row[0];
    Out high = row[1];
    for (int g = 1; g < num_devices; g++)
    {
      low = std::min(low, row[2 * g]);
      high = std::max(high, row[2 * g + 1]);
    }
    if (out_min != nullptr)
    {
      out_min[k] = low;
    }
    if (out_max != nullptr)
    {
      out_max[k] = high;
    }
  }
}

// 1..8 distinct devices.
int CheckDeviceList(const int* devices, int num_devices)
{
  if (devices == nullptr || num_devices < 1 || num_devices > 8)
  {
    return FailInvalid("1..8 devices are supported");
  }
  for (int a = 0; a < num_devices; a++)
  {
    for (int b = a + 1; b < num_devices; b++)
    {
      if (devices[a] == devices[b])
      {
        return FailInvalid("device %d is listed twice", devices[a]);
      }
    }
  }
  return VGT_B200_OK;
}

// The cell and double entries also refuse an ordinal outside [0, 64) (the receive-buffer cache's
// range) before any device call.
int CheckMultiDeviceList(const int* devices, int num_devices, int64_t nx, int64_t ny)
{
  const int check = CheckDeviceList(devices, num_devices);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  for (int g = 0; g < num_devices; g++)
  {
    if (devices[g] < 0 || devices[g] >= 64)
    {
      return FailInvalid("device ordinal %d out of range", devices[g]);
    }
  }
  if (num_devices > 1 && (num_devices > nx || num_devices > ny))
  {
    return FailInvalid("more devices than voxels along x or y");
  }
  return VGT_B200_OK;
}

// The driver of every multi-device entry. Work supplies the per-slab steps:
//   typename Work::Slab                      per-device state, built on that device's thread
//   int Local(Slab&, const SlabPart&, r)     enqueue the input of round r and the local passes
//                                            (ExchangeLocalPasses)
//   bool FinalMinMax(r)                      whether the final pass of round r reduces min/max
//   int Emit(Slab&, const SlabPart&, r, Out* const* d_slabs, Out* d_min_max)
//                                            what becomes of the y-slab of round r
//   int slab_buffers                         y-slabs kept (round r writes d_slabs[r % count])
// The driver synchronises the stream after Local and after Emit.
template <int kMode, typename Work>
int SdfMultiDevice(const MultiGrid& grid, const int* devices, int64_t rounds, const Work& job)
{
  using Out = typename OutputOf<kMode>::Type;
  const int num_devices = grid.num_devices;
  // Peer access between every pair (a one-time, process-wide driver setting; "already enabled"
  // is fine). Without it the fused exchange cannot run: no silent fallback.
  for (int a = 0; a < num_devices; a++)
  {
    ScopedDevice scoped(devices[a]);
    VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
    for (int b = 0; b < num_devices; b++)
    {
      if (a == b)
      {
        continue;
      }
      int can_access = 0;
      VGT_CUDA_TRY(cudaDeviceCanAccessPeer(&can_access, devices[a], devices[b]), "peer query");
      if (can_access == 0)
      {
        SetLastError("device %d cannot access device %d as a peer", devices[a], devices[b]);
        return VGT_B200_ERR_DEVICE;
      }
      const cudaError_t enabled = cudaDeviceEnablePeerAccess(devices[b], 0);
      if (enabled != cudaSuccess && enabled != cudaErrorPeerAccessAlreadyEnabled)
      {
        return FailDevice("cudaDeviceEnablePeerAccess", enabled);
      }
      cudaGetLastError();
    }
  }
  const int64_t widest_part = (grid.ny + num_devices - 1) / num_devices;
  const int64_t receive_words = grid.nx * widest_part * grid.nz;
  // Receive buffers: plain cudaMalloc (peer-mapped once access is enabled; pool memory would
  // need per-pool access grants). cudaMalloc / cudaFree of half a gigabyte per device and call
  // costs more than the passes, so one buffer per device is kept for the life of the process
  // and grows on demand; a call holds the cache lock while it uses them (multi-device calls of
  // one process run one at a time).
  static std::mutex receive_mutex;
  static uint32_t* cached_buffer[64] = {};
  static size_t cached_words[64] = {};
  std::lock_guard<std::mutex> receive_lock(receive_mutex);
  std::vector<uint32_t*> receive(static_cast<size_t>(num_devices), nullptr);
  for (int g = 0; g < num_devices; g++)
  {
    const int device = devices[g];
    if (device < 0 || device >= 64)
    {
      return FailInvalid("device ordinal %d out of range", device);
    }
    ScopedDevice scoped(device);
    VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
    if (cached_words[device] < static_cast<size_t>(receive_words))
    {
      if (cached_buffer[device] != nullptr)
      {
        cudaFree(cached_buffer[device]);
        cached_buffer[device] = nullptr;
        cached_words[device] = 0;
      }
      VGT_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&cached_buffer[device]),
                              sizeof(uint32_t) * static_cast<size_t>(receive_words)),
                   "receive buffer allocation");
      cached_words[device] = static_cast<size_t>(receive_words);
    }
    receive[static_cast<size_t>(g)] = cached_buffer[device];
  }
  std::vector<uint64_t> peer_bases(static_cast<size_t>(num_devices));
  for (int g = 0; g < num_devices; g++)
  {
    peer_bases[static_cast<size_t>(g)] = reinterpret_cast<uint64_t>(receive[static_cast<size_t>(g)]);
  }

  ThreadBarrier barrier(num_devices);
  std::vector<int> statuses(static_cast<size_t>(num_devices), VGT_B200_OK);
  std::vector<std::string> messages(static_cast<size_t>(num_devices));
  std::atomic<int> failed{0};

  const auto worker = [&](const int g)
  {
    int status = VGT_B200_OK;
    const int device = devices[g];
    ScopedDevice scoped(device);
    SlabPart part{};
    part.index = g;
    SplitRange(grid.nx, num_devices, g, &part.x0, &part.x1);
    SplitRange(grid.ny, num_devices, g, &part.y0, &part.y1);
    part.peer_bases = peer_bases.data();
    StreamGuard guard;
    StreamScratch<uint32_t> d_scratch;
    StreamScratch<Out> d_slabs[2];
    StreamScratch<Out> d_min_max;
    typename Work::Slab slab;
    StagedTransfer transfer;
    if (num_devices >= 6)
    {
      // enough device threads to be the parallel copy workers themselves (the shared workers
      // serve one caller at a time); with fewer devices the shared workers copy faster
      transfer.UseCallingThreadOnly();
    }
    part.transfer = &transfer;
    // (runs first on every exit path: nothing is queued when the buffers are released)
    struct DrainOnExit
    {
      const StreamGuard& guard;
      ~DrainOnExit()
      {
        if (guard.stream != nullptr)
        {
          cudaStreamSynchronize(guard.stream);
        }
      }
    } drain{guard};
    const auto local_passes = [&](int64_t round) -> int
    {
      if (round == 0)
      {
        VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
        KeepPoolMemory(device);
        VGT_CUDA_TRY(cudaStreamCreateWithFlags(&guard.stream, cudaStreamNonBlocking), "stream");
        part.stream = guard.stream;
        VGT_CUDA_TRY(d_scratch.Allocate(part.Voxels(grid), part.stream),
                     "local pass scratch allocation");
        part.scratch = d_scratch.get();
      }
      const int local = job.Local(slab, part, round);
      if (local != VGT_B200_OK)
      {
        return local;
      }
      VGT_CUDA_TRY(cudaStreamSynchronize(part.stream), "slab-local passes");
      return VGT_B200_OK;
    };
    const auto final_pass = [&](int64_t round) -> int
    {
      const int64_t rows = part.y1 - part.y0;
      StreamScratch<Out>& target = d_slabs[round % job.slab_buffers];
      if (target.get() == nullptr)
      {
        VGT_CUDA_TRY(target.Allocate(grid.nx * rows * grid.nz, part.stream),
                     "SDF slab allocation");
      }
      if (d_min_max.get() == nullptr)
      {
        VGT_CUDA_TRY(d_min_max.Allocate(2, part.stream), "min/max allocation");
      }
      const int final_status = RunFinalPass<kMode>(
          receive[static_cast<size_t>(g)], grid.nx, rows, grid.nz, part.y0, grid.ny,
          grid.resolution, grid.add_virtual_border, target.get(),
          job.FinalMinMax(round) ? d_min_max.get() : nullptr, part.stream);
      if (final_status != VGT_B200_OK)
      {
        return final_status;
      }
      Out* const slabs[2] = {d_slabs[0].get(), d_slabs[1].get()};
      const int emitted = job.Emit(slab, part, round, slabs, d_min_max.get());
      if (emitted != VGT_B200_OK)
      {
        return emitted;
      }
      VGT_CUDA_TRY(cudaStreamSynchronize(part.stream), "SDF generation");
      return VGT_B200_OK;
    };
    const auto fail = [&](int code)
    {
      status = code;
      messages[static_cast<size_t>(g)] = vgt_b200_last_error();  // thread-local text
      failed.store(1);
    };
    const auto stand_down = [&]()
    {
      status = VGT_B200_ERR_DEVICE;
      messages[static_cast<size_t>(g)] = "another device failed";
    };
    // Every thread reaches every barrier, whatever has failed before.
    for (int64_t round = 0; round < rounds; round++)
    {
      if (status == VGT_B200_OK && failed.load() != 0)
      {
        stand_down();
      }
      if (status == VGT_B200_OK)
      {
        const int local = local_passes(round);
        if (local != VGT_B200_OK)
        {
          fail(local);
        }
      }
      // every device's stores into every receive buffer have landed
      barrier.Wait();
      if (status == VGT_B200_OK && failed.load() != 0)
      {
        stand_down();
      }
      else if (status == VGT_B200_OK)
      {
        const int final_status = final_pass(round);
        if (final_status != VGT_B200_OK)
        {
          fail(final_status);
        }
      }
      // The exchange of round r + 1 stores into the other devices' receive buffers, which their
      // final pass of round r reads. One receive buffer per device and this barrier, rather than
      // two buffers used alternately: the receive buffer is the largest allocation after the
      // cells, and final_pass has drained its stream (the copy-out waits for it anyway), so the
      // barrier costs no more than the slowest device's final pass.
      if (round + 1 < rounds)
      {
        barrier.Wait();
      }
    }
    statuses[static_cast<size_t>(g)] = status;
  };
  std::vector<std::thread> threads;
  for (int g = 1; g < num_devices; g++)
  {
    threads.emplace_back(worker, g);
  }
  worker(0);
  for (auto& thread : threads)
  {
    thread.join();
  }
  // the device that failed first-hand, not the ones that stood down because of it
  for (const bool first_hand : {true, false})
  {
    for (int g = 0; g < num_devices; g++)
    {
      const bool stood_down = messages[static_cast<size_t>(g)] == "another device failed";
      if (statuses[static_cast<size_t>(g)] != VGT_B200_OK && stood_down != first_hand)
      {
        SetLastError("device %d: %s", devices[g], messages[static_cast<size_t>(g)].c_str());
        return statuses[static_cast<size_t>(g)];
      }
    }
  }
  return VGT_B200_OK;
}

// OccupancyMap: the float occupancy slab, one round.
template <int kMode>
struct OccupancySlabs
{
  using Out = typename OutputOf<kMode>::Type;
  struct Slab
  {
    StreamScratch<float> occupancy;
  };
  MultiGrid grid;
  const float* h_in;
  int unknown_is_filled;
  Out* h_out;
  mutable std::vector<Out> extrema;  // [device][min, max]
  int slab_buffers = 1;

  int Local(Slab& slab, const SlabPart& part, int64_t) const
  {
    const int64_t voxels = part.Voxels(grid);
    VGT_CUDA_TRY(slab.occupancy.Allocate(voxels, part.stream), "occupancy slab allocation");
    const size_t bytes = sizeof(float) * static_cast<size_t>(voxels);
    VGT_CUDA_TRY(part.transfer->ToDevice(reinterpret_cast<char*>(slab.occupancy.get()), bytes,
                                         reinterpret_cast<const char*>(h_in
                                                                       + part.x0 * grid.Plane()),
                                         bytes, bytes, 1, part.stream),
                 "copy occupancy slab to device");
    return ExchangeLocalPasses<float>(slab.occupancy.get(), unknown_is_filled, grid, part);
  }
  bool FinalMinMax(int64_t) const { return true; }
  int Emit(Slab&, const SlabPart& part, int64_t, Out* const* d_slabs, Out* d_min_max) const
  {
    return CopySlabToHost(d_slabs[0], d_min_max, grid, part, h_out,
                          extrema.data() + 2 * part.index);
  }
};

template <int kMode>
int SdfOccupancyMultiDevice(const float* h_in, int64_t nx, int64_t ny, int64_t nz,
                            double resolution, int unknown_is_filled, int add_virtual_border,
                            const int* devices, int num_devices,
                            typename OutputOf<kMode>::Type* h_out,
                            typename OutputOf<kMode>::Type* out_min,
                            typename OutputOf<kMode>::Type* out_max)
{
  const int check = CheckSdfArguments(h_in, h_out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  const int listed = CheckDeviceList(devices, num_devices);
  if (listed != VGT_B200_OK)
  {
    return listed;
  }
  if (num_devices == 1)
  {
    return SdfFromHost<float, kMode>(h_in, nx, ny, nz, resolution, unknown_is_filled,
                                     add_virtual_border, devices[0], h_out, out_min, out_max);
  }
  if (num_devices > nx || num_devices > ny)
  {
    return FailInvalid("more devices than voxels along x or y");
  }
  OccupancySlabs<kMode> job{};
  job.grid = MultiGrid{nx, ny, nz, resolution, add_virtual_border, num_devices};
  job.h_in = h_in;
  job.unknown_is_filled = unknown_is_filled;
  job.h_out = h_out;
  job.extrema.resize(2 * static_cast<size_t>(num_devices));
  const int status = SdfMultiDevice<kMode>(job.grid, devices, 1, job);
  if (status != VGT_B200_OK)
  {
    return status;
  }
  CombineExtrema(job.extrema, num_devices, 1, out_min, out_max);
  return VGT_B200_OK;
}

enum CellMember
{
  kCellSdf = 0,        // the objects_to_use SDF
  kCellFreeAndNamed = 1,
  kCellPerObject = 2   // MakeSeparateObjectSDFs
};

// The three cell-map members: the cell slab is uploaded in round 0 and stays resident.
//   kCellSdf:          one round on the filled mask (CellsToMaskKernel with the sorted id list).
//   kCellFreeAndNamed: round 0 on all filled cells, round 1 on the filled cells of named objects
//                      (id > 0); both y-slabs are kept and merged elementwise, which is exact on
//                      a y-slab.
//   kCellPerObject:    one round per listed id, in the order of the id's sorted position so that
//                      each group of kSlotGroupSize distinct ids is classified once per slab
//                      (CellsToObjectSlotsKernel); round r runs the z scan on "slot == key".
template <int kMode>
struct CellSlabs
{
  using Out = typename OutputOf<kMode>::Type;
  using Key = typename OutputOf<kMode>::Key;
  struct Slab
  {
    StreamScratch<uint32_t> cells;
    StreamScratch<uint8_t> mask;  // the filled mask, or the slot map of the batch
    StreamScratch<uint32_t> ids;
    StreamScratch<Key> keys;
    int64_t group = -1;           // the slot group `mask` holds
  };
  MultiGrid grid;
  CellMember member;
  const void* h_cells;
  int cell_bytes;
  int unknown_is_filled;
  std::vector<uint32_t> sorted;    // distinct ids, ascending
  std::vector<int64_t> position;   // kCellPerObject: index of object_ids[k] in `sorted`
  std::vector<int64_t> order;      // kCellPerObject: round -> k
  Out* h_out;
  mutable std::vector<Out> extrema;  // [result][device][min, max]
  int slab_buffers = 1;

  int Local(Slab& slab, const SlabPart& part, int64_t round) const
  {
    const int64_t voxels = part.Voxels(grid);
    const int cell_words = cell_bytes / 4;
    if (round == 0)
    {
      VGT_CUDA_TRY(slab.cells.Allocate(voxels * cell_words, part.stream),
                   "cell slab allocation");
      VGT_CUDA_TRY(slab.mask.Allocate(voxels, part.stream), "filled mask allocation");
      const size_t bytes = static_cast<size_t>(voxels) * cell_bytes;
      const char* source = static_cast<const char*>(h_cells)
          + static_cast<size_t>(part.x0 * grid.Plane()) * cell_bytes;
      VGT_CUDA_TRY(part.transfer->ToDevice(reinterpret_cast<char*>(slab.cells.get()), bytes,
                                           source, bytes, bytes, 1, part.stream),
                   "copy cell slab to device");
      if (member == kCellSdf)
      {
        const int uploaded = UploadIds(sorted, slab.ids, part.stream);
        if (uploaded != VGT_B200_OK)
        {
          return uploaded;
        }
      }
    }
    const int threads = 256;
    if (member == kCellPerObject)
    {
      const int64_t slot = position[static_cast<size_t>(order[static_cast<size_t>(round)])];
      const int64_t group = slot / kSlotGroupSize;
      if (group != slab.group)
      {
        SlotGroup ids{};
        const int64_t first = group * kSlotGroupSize;
        ids.count = static_cast<int>(
            std::min<int64_t>(kSlotGroupSize, static_cast<int64_t>(sorted.size()) - first));
        std::copy(sorted.begin() + first, sorted.begin() + first + ids.count, ids.ids);
        const int64_t blocks = std::min<int64_t>((voxels + threads * 4 - 1) / (threads * 4),
                                                 MultiprocessorCount() * 8);
        CellsToObjectSlotsKernel<<<static_cast<unsigned>(blocks), threads, 0, part.stream>>>(
            slab.cells.get(), cell_words, voxels, unknown_is_filled, ids, slab.mask.get()); NoteKernelLaunch();
        VGT_CUDA_TRY(cudaGetLastError(), "CellsToObjectSlotsKernel launch");
        slab.group = group;
      }
      const int key = static_cast<int>(slot % kSlotGroupSize) + 1;
      return ExchangeLocalPasses<ObjectSlot>(reinterpret_cast<const ObjectSlot*>(slab.mask.get()),
                                             key, grid, part);
    }
    int rule = kAnyObject;
    if (member == kCellSdf && !sorted.empty())
    {
      rule = kListedObjects;
    }
    else if (member == kCellFreeAndNamed && round == 1)
    {
      rule = kNamedObjects;
    }
    const int num_ids = (rule == kListedObjects) ? static_cast<int>(sorted.size()) : 0;
    CellsToMaskKernel<<<static_cast<unsigned>((voxels + threads - 1) / threads), threads, 0,
                        part.stream>>>(slab.cells.get(), cell_words, voxels, unknown_is_filled,
                                       rule, num_ids > 0 ? slab.ids.get() : nullptr, num_ids,
                                       slab.mask.get()); NoteKernelLaunch();
    VGT_CUDA_TRY(cudaGetLastError(), "CellsToMaskKernel launch");
    return ExchangeLocalPasses<uint8_t>(slab.mask.get(), 0, grid, part);
  }
  bool FinalMinMax(int64_t) const { return member != kCellFreeAndNamed; }
  int Emit(Slab& slab, const SlabPart& part, int64_t round, Out* const* d_slabs,
           Out* d_min_max) const
  {
    const int64_t count = grid.nx * grid.ny * grid.nz;
    if (member == kCellSdf)
    {
      return CopySlabToHost(d_slabs[0], d_min_max, grid, part, h_out,
                            extrema.data() + 2 * part.index);
    }
    if (member == kCellPerObject)
    {
      const int64_t k = order[static_cast<size_t>(round)];
      return CopySlabToHost(d_slabs[0], d_min_max, grid, part, h_out + k * count,
                            extrema.data() + 2 * (k * grid.num_devices + part.index));
    }
    if (round == 0)
    {
      return VGT_B200_OK;  // the all-filled y-slab waits in d_slabs[0] for the named one
    }
    // SdfFreeAndNamedOnDevice's merge on the y-slab: d_slabs[0] = merge(free, named)
    const int64_t slab_voxels = grid.nx * (part.y1 - part.y0) * grid.nz;
    if (slab.keys.get() == nullptr)
    {
      VGT_CUDA_TRY(slab.keys.Allocate(2, part.stream), "min/max scratch");
    }
    ResetMinMaxKeysKernel<Key><<<1, 1, 0, part.stream>>>(slab.keys.get()); NoteKernelLaunch();
    const int threads = 256;
    const int64_t merge_blocks =
        std::min<int64_t>((slab_voxels + threads - 1) / threads, MultiprocessorCount() * 16);
    MergeFreeAndNamedKernel<Out, Key>
        <<<static_cast<unsigned>(merge_blocks), threads, 0, part.stream>>>(
            d_slabs[0], d_slabs[1], slab_voxels, d_slabs[0], slab.keys.get()); NoteKernelLaunch();
    DecodeMinMaxKernel<Out, Key><<<1, 1, 0, part.stream>>>(slab.keys.get(), d_min_max); NoteKernelLaunch();
    VGT_CUDA_TRY(cudaGetLastError(), "MergeFreeAndNamedKernel launch");
    return CopySlabToHost(d_slabs[0], d_min_max, grid, part, h_out,
                          extrema.data() + 2 * part.index);
  }
};

template <int kMode>
int SdfCellsMultiDevice(CellMember member, const void* h_cells, int cell_bytes, int64_t nx,
                        int64_t ny, int64_t nz, double resolution, int unknown_is_filled,
                        int add_virtual_border, const uint32_t* object_ids,
                        int64_t num_object_ids, const int* devices, int num_devices,
                        typename OutputOf<kMode>::Type* h_out,
                        typename OutputOf<kMode>::Type* out_min,
                        typename OutputOf<kMode>::Type* out_max)
{
  using Out = typename OutputOf<kMode>::Type;
  if (member == kCellFreeAndNamed)
  {
    object_ids = nullptr;
    num_object_ids = 0;
  }
  const int check = CheckCellArguments(h_cells, cell_bytes, h_out, nx, ny, nz, resolution,
                                       object_ids, num_object_ids);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  const int listed = CheckMultiDeviceList(devices, num_devices, nx, ny);
  if (listed != VGT_B200_OK)
  {
    return listed;
  }
  const int64_t count = nx * ny * nz;
  if (member == kCellPerObject && num_object_ids > 0
      && count * static_cast<int64_t>(sizeof(Out)) > INT64_MAX / num_object_ids)
  {
    return FailInvalid("%lld SDFs of %lld voxels overflow a 64-bit byte count",
                       static_cast<long long>(num_object_ids), static_cast<long long>(count));
  }
  if (num_devices == 1)
  {
    if (member == kCellFreeAndNamed)
    {
      return SdfFreeAndNamedHost<kMode>(h_cells, cell_bytes, nx, ny, nz, resolution,
                                        unknown_is_filled, add_virtual_border, devices[0], h_out,
                                        out_min, out_max);
    }
    return SdfFromCellsHost<kMode>(h_cells, cell_bytes, nx, ny, nz, resolution,
                                   unknown_is_filled, add_virtual_border, object_ids,
                                   num_object_ids, member == kCellPerObject, devices[0], h_out,
                                   out_min, out_max);
  }
  // (every device answers before the id list is read; an empty batch launches nothing, but it
  // still needs the devices it was asked to use)
  for (int g = 0; g < num_devices; g++)
  {
    ScopedDevice scoped(devices[g]);
    VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  }
  if (member == kCellPerObject && num_object_ids == 0)
  {
    return VGT_B200_OK;
  }
  CellSlabs<kMode> job{};
  job.grid = MultiGrid{nx, ny, nz, resolution, add_virtual_border, num_devices};
  job.member = member;
  job.h_cells = h_cells;
  job.cell_bytes = cell_bytes;
  job.unknown_is_filled = unknown_is_filled;
  job.h_out = h_out;
  job.sorted = SortedDistinct(object_ids, num_object_ids);
  int64_t rounds = 1;
  int64_t results = 1;
  if (member == kCellFreeAndNamed)
  {
    rounds = 2;
    job.slab_buffers = 2;
  }
  else if (member == kCellPerObject)
  {
    rounds = results = num_object_ids;
    job.position.resize(static_cast<size_t>(num_object_ids));
    job.order.resize(static_cast<size_t>(num_object_ids));
    for (int64_t k = 0; k < num_object_ids; k++)
    {
      job.position[static_cast<size_t>(k)] =
          std::lower_bound(job.sorted.begin(), job.sorted.end(), object_ids[k])
          - job.sorted.begin();
      job.order[static_cast<size_t>(k)] = k;
    }
    std::stable_sort(job.order.begin(), job.order.end(), [&](int64_t a, int64_t b)
    {
      return job.position[static_cast<size_t>(a)] < job.position[static_cast<size_t>(b)];
    });
  }
  job.extrema.resize(2 * static_cast<size_t>(results * num_devices));
  const int status = SdfMultiDevice<kMode>(job.grid, devices, rounds, job);
  if (status != VGT_B200_OK)
  {
    return status;
  }
  CombineExtrema(job.extrema, num_devices, results, out_min, out_max);
  return VGT_B200_OK;
}

// ComputeDistanceFieldTransformInPlace on a host double field: see edt_transform.cuh.
int TransformFieldInPlace(double* h_field, int64_t nx, int64_t ny, int64_t nz)
{
  const int64_t count = nx * ny * nz;
  StreamGuard guard;
  VGT_CUDA_TRY(cudaStreamCreateWithFlags(&guard.stream, cudaStreamNonBlocking),
               "cudaStreamCreate");
  cudaStream_t stream = guard.stream;
  StreamScratch<double> d_field;
  StreamScratch<uint32_t> d_a;
  StreamScratch<uint32_t> d_b;
  StreamScratch<uint32_t> d_report;
  VGT_CUDA_TRY(d_field.Allocate(count, stream), "field allocation");
  VGT_CUDA_TRY(d_a.Allocate(count, stream), "packed field allocation");
  VGT_CUDA_TRY(d_b.Allocate(count, stream), "packed field allocation");
  VGT_CUDA_TRY(d_report.Allocate(2, stream), "ingest report allocation");
  VGT_CUDA_TRY(cudaMemsetAsync(d_report.get(), 0, sizeof(uint32_t) * 2, stream), "report reset");
  VGT_CUDA_TRY(cudaMemcpyAsync(d_field.get(), h_field, sizeof(double) * count,
                               cudaMemcpyHostToDevice, stream),
               "copy field to device");
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((count + threads - 1) / threads);
  IngestSamplesKernel<<<blocks, threads, 0, stream>>>(d_field.get(), count, d_a.get(),
                                                      d_report.get()); NoteKernelLaunch();
  uint32_t report[2] = {0u, 0u};
  VGT_CUDA_TRY(cudaMemcpyAsync(report, d_report.get(), sizeof(report), cudaMemcpyDeviceToHost,
                               stream),
               "copy ingest report");
  VGT_CUDA_TRY(cudaStreamSynchronize(stream), "field ingest");
  if (report[0] != 0u)
  {
    SetLastError("%u samples are neither +inf nor a non-negative integer below 2^31 - 1 (the "
                 "device transform is exact integer arithmetic)", report[0]);
    return VGT_B200_ERR_UNSUPPORTED;
  }
  const int64_t largest = static_cast<int64_t>(report[1]) + Square(nx - 1) + Square(ny - 1)
      + Square(nz - 1);
  if (largest > kLeanMaxInput)
  {
    SetLastError("samples up to %u on a %lld x %lld x %lld grid exceed the 2^29 range of the "
                 "integer passes", report[1], static_cast<long long>(nx),
                 static_cast<long long>(ny), static_cast<long long>(nz));
    return VGT_B200_ERR_UNSUPPORTED;
  }
  // Pass order X, Y, Z as the reference (sdfgen.cpp:276-390); an axis of one voxel is skipped.
  uint32_t* front = d_a.get();
  uint32_t* back = d_b.get();
  int64_t max_input = report[1];
  if (nx > 1)
  {
    const int status = LaunchEnvelope<kEmitPacked>(front, back, FamilyAlongX(nx, ny, nz),
                                                   max_input, FinalizeParams{}, nullptr, stream);
    if (status != VGT_B200_OK)
    {
      return status;
    }
    std::swap(front, back);
    max_input += Square(nx - 1);
  }
  if (ny > 1)
  {
    const int status = LaunchEnvelope<kEmitPacked>(front, back, FamilyAlongY(nx, ny, nz),
                                                   max_input, FinalizeParams{}, nullptr, stream);
    if (status != VGT_B200_OK)
    {
      return status;
    }
    std::swap(front, back);
    max_input += Square(ny - 1);
  }
  if (nz > 1)
  {
    // [nx][ny][nz] -> [nx][nz][ny], lines along the (now strided) z axis, and back
    const dim3 tile(32, 8);
    TransposePlanesKernel<<<dim3(static_cast<unsigned>((nz + 31) / 32),
                                 static_cast<unsigned>((ny + 31) / 32),
                                 static_cast<unsigned>(nx)),
                            tile, 0, stream>>>(front, back, static_cast<int>(ny),
                                               static_cast<int>(nz)); NoteKernelLaunch();
    const int status = LaunchEnvelope<kEmitPacked>(back, front, FamilyAlongY(nx, nz, ny),
                                                   max_input, FinalizeParams{}, nullptr, stream);
    if (status != VGT_B200_OK)
    {
      return status;
    }
    TransposePlanesKernel<<<dim3(static_cast<unsigned>((ny + 31) / 32),
                                 static_cast<unsigned>((nz + 31) / 32),
                                 static_cast<unsigned>(nx)),
                            tile, 0, stream>>>(front, back, static_cast<int>(nz),
                                               static_cast<int>(ny)); NoteKernelLaunch();
    std::swap(front, back);
  }
  EmitSamplesKernel<<<blocks, threads, 0, stream>>>(front, count, d_field.get()); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "transform kernels");
  VGT_CUDA_TRY(cudaMemcpyAsync(h_field, d_field.get(), sizeof(double) * count,
                               cudaMemcpyDeviceToHost, stream),
               "copy field to host");
  VGT_CUDA_TRY(cudaStreamSynchronize(stream), "distance field transform");
  return VGT_B200_OK;
}
}  // namespace
}  // namespace edt
}  // namespace vgt_b200

// ================================================================================================
// C-ABI (include/vgt_b200.h)
// ================================================================================================
using namespace vgt_b200;
using namespace vgt_b200::edt;

extern "C"
{
int vgt_b200_sdf_f32_dev(
    const float* d_occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* d_sdf_out, float* d_min_max,
    void* stream)
{
  const int check = CheckSdfArguments(d_occupancy, d_sdf_out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  return SdfOnDevice<float, kEmitFloat>(d_occupancy, nx, ny, nz, resolution, unknown_is_filled,
                                        add_virtual_border, d_sdf_out, d_min_max,
                                        static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_f32_dev_profile(
    const float* d_occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* d_sdf_out, float* d_min_max,
    void* stream, float* out_pass_ms)
{
  const int check = CheckSdfArguments(d_occupancy, d_sdf_out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (out_pass_ms == nullptr)
  {
    return FailInvalid("null out_pass_ms");
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaEvent_t marks[4];
  for (auto& mark : marks)
  {
    VGT_CUDA_TRY(cudaEventCreate(&mark), "cudaEventCreate");
  }
  WindowKernelMarks window_marks;
  for (int i = 0; i < 2; i++)
  {
    VGT_CUDA_TRY(cudaEventCreate(&window_marks.begin[i]), "cudaEventCreate");
    VGT_CUDA_TRY(cudaEventCreate(&window_marks.end[i]), "cudaEventCreate");
  }
  g_window_marks = &window_marks;
  const int status =
      SdfOnDevice<float, kEmitFloat>(d_occupancy, nx, ny, nz, resolution, unknown_is_filled,
                                     add_virtual_border, d_sdf_out, d_min_max, s, marks);
  g_window_marks = nullptr;
  const cudaError_t sync = cudaStreamSynchronize(s);
  out_pass_ms[3] = 0.0f;
  out_pass_ms[4] = 0.0f;
  if (status == VGT_B200_OK && sync == cudaSuccess)
  {
    for (int i = 0; i < 3; i++)
    {
      cudaEventElapsedTime(out_pass_ms + i, marks[i], marks[i + 1]);
    }
    // (a grid with a one-voxel axis skips that pass: the launches are then fewer than two, and
    // the first one belongs to whichever strided pass ran)
    for (int i = 0; i < window_marks.launches; i++)
    {
      const int slot = (window_marks.launches == 2) ? 3 + i : (ny > 1 ? 3 : 4);
      cudaEventElapsedTime(out_pass_ms + slot, window_marks.begin[i], window_marks.end[i]);
    }
  }
  for (auto& mark : marks)
  {
    cudaEventDestroy(mark);
  }
  for (int i = 0; i < 2; i++)
  {
    cudaEventDestroy(window_marks.begin[i]);
    cudaEventDestroy(window_marks.end[i]);
  }
  if (status != VGT_B200_OK)
  {
    return status;
  }
  VGT_CUDA_TRY(sync, "profiled SDF generation");
  return VGT_B200_OK;
}

int vgt_b200_sdf_from_mask_f32_dev(
    const uint8_t* d_filled_mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int add_virtual_border, int device, float* d_sdf_out, float* d_min_max, void* stream)
{
  const int check = CheckSdfArguments(d_filled_mask, d_sdf_out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  return SdfOnDevice<uint8_t, kEmitFloat>(d_filled_mask, nx, ny, nz, resolution, 0,
                                          add_virtual_border, d_sdf_out, d_min_max,
                                          static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_f64_dev(
    const float* d_occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* d_sdf_out,
    double* d_min_max, void* stream)
{
  const int check = CheckSdfArguments(d_occupancy, d_sdf_out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  return SdfOnDevice<float, kEmitDouble>(d_occupancy, nx, ny, nz, resolution, unknown_is_filled,
                                         add_virtual_border, d_sdf_out, d_min_max,
                                         static_cast<cudaStream_t>(stream));
}

int vgt_b200_edt_local_passes_dev(
    const float* d_occupancy, int64_t nx_local, int64_t ny, int64_t nz, int unknown_is_filled,
    int send_parts, int device, int32_t* d_out, void* stream)
{
  const int check = CheckSdfArguments(d_occupancy, d_out, nx_local, ny, nz, 1.0);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (send_parts < 0)
  {
    return FailInvalid("send_parts must be >= 0");
  }
  StreamScratch<uint32_t> scratch;
  if (ny > 1 || send_parts > 1)
  {
    VGT_CUDA_TRY(scratch.Allocate(nx_local * ny * nz, s), "local pass scratch allocation");
  }
  return RunLocalPasses<float>(d_occupancy, nx_local, ny, nz, unknown_is_filled,
                               reinterpret_cast<uint32_t*>(d_out), scratch.get(), s, send_parts);
}

int vgt_b200_edt_local_passes_scatter_dev(
    const float* d_occupancy, int64_t nx_local, int64_t ny, int64_t nz, int unknown_is_filled,
    int num_ranks, int rank, int64_t x_offset, int64_t nx_total,
    const uint64_t* peer_receive_buffers, int64_t receive_capacity_words, int device, void* stream)
{
  const int check = CheckSdfArguments(d_occupancy, peer_receive_buffers, nx_local, ny, nz, 1.0);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (num_ranks < 2 || num_ranks > 8 || rank < 0 || rank >= num_ranks)
  {
    return FailInvalid("fused exchange needs 2..8 ranks and a rank inside that range");
  }
  if (x_offset < 0 || nx_total > VGT_B200_MAX_AXIS || x_offset + nx_local > nx_total)
  {
    return FailInvalid("x slab [%lld, %lld) does not fit nx_total = %lld",
                       static_cast<long long>(x_offset),
                       static_cast<long long>(x_offset + nx_local),
                       static_cast<long long>(nx_total));
  }
  // the largest part of a y line is ceil(ny / num_ranks) rows: every receive buffer must hold
  // [nx_total][that many rows][nz] words, or a peer store would land outside it
  const int64_t widest_part = (ny + num_ranks - 1) / num_ranks;
  if (receive_capacity_words < nx_total * widest_part * nz)
  {
    return FailInvalid("receive buffers of %lld words cannot hold %lld x %lld x %lld",
                       static_cast<long long>(receive_capacity_words),
                       static_cast<long long>(nx_total), static_cast<long long>(widest_part),
                       static_cast<long long>(nz));
  }
  for (int peer = 0; peer < num_ranks; peer++)
  {
    if (peer_receive_buffers[peer] == 0)
    {
      return FailInvalid("null peer receive buffer %d", peer);
    }
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  StreamScratch<uint32_t> scratch;
  VGT_CUDA_TRY(scratch.Allocate(nx_local * ny * nz, s), "local pass scratch allocation");
  // d_result is unused in scatter mode (every part has a remote or self-mapped destination).
  return RunLocalPasses<float>(d_occupancy, nx_local, ny, nz, unknown_is_filled, scratch.get(),
                               scratch.get(), s, num_ranks, peer_receive_buffers, x_offset, rank);
}

int vgt_b200_edt_final_pass_f32_dev(
    int32_t* d_in, int64_t nx, int64_t ny_local, int64_t nz, int64_t y_offset, int64_t ny_total,
    double resolution, int add_virtual_border, int device, float* d_sdf_out, float* d_min_max,
    void* stream)
{
  const int check = CheckSdfArguments(d_in, d_sdf_out, nx, ny_local, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (static_cast<const void*>(d_in) == static_cast<const void*>(d_sdf_out))
  {
    return FailInvalid("d_in and d_sdf_out must not alias");
  }
  if (y_offset < 0 || ny_total < 1 || ny_total > VGT_B200_MAX_AXIS
      || y_offset + ny_local > ny_total)
  {
    return FailInvalid("y slab [%lld, %lld) does not fit ny_total = %lld",
                       static_cast<long long>(y_offset),
                       static_cast<long long>(y_offset + ny_local),
                       static_cast<long long>(ny_total));
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  return RunFinalPass<kEmitFloat>(reinterpret_cast<uint32_t*>(d_in), nx, ny_local, nz, y_offset,
                                  ny_total, resolution, add_virtual_border, d_sdf_out, d_min_max,
                                  static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_f32(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* sdf_out, float* out_min,
    float* out_max)
{
  return SdfFromHost<float, kEmitFloat>(occupancy, nx, ny, nz, resolution, unknown_is_filled,
                                        add_virtual_border, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_f32_multi(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max)
{
  return SdfOccupancyMultiDevice<kEmitFloat>(occupancy, nx, ny, nz, resolution,
                                             unknown_is_filled, add_virtual_border, devices,
                                             num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_f64_multi(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max)
{
  const int check = CheckSdfArguments(occupancy, sdf_out, nx, ny, nz, resolution);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  const int listed = CheckMultiDeviceList(devices, num_devices, nx, ny);
  if (listed != VGT_B200_OK)
  {
    return listed;
  }
  return SdfOccupancyMultiDevice<kEmitDouble>(occupancy, nx, ny, nz, resolution,
                                              unknown_is_filled, add_virtual_border, devices,
                                              num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_f64(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* sdf_out, double* out_min,
    double* out_max)
{
  return SdfFromHost<float, kEmitDouble>(occupancy, nx, ny, nz, resolution, unknown_is_filled,
                                         add_virtual_border, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_from_mask_f32(
    const uint8_t* filled_mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int add_virtual_border, int device, float* sdf_out, float* out_min, float* out_max)
{
  return SdfFromHost<uint8_t, kEmitFloat>(filled_mask, nx, ny, nz, resolution, 0,
                                          add_virtual_border, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_from_mask_f64(
    const uint8_t* filled_mask, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int add_virtual_border, int device, double* sdf_out, double* out_min, double* out_max)
{
  return SdfFromHost<uint8_t, kEmitDouble>(filled_mask, nx, ny, nz, resolution, 0,
                                           add_virtual_border, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_from_cells_f32(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* sdf_out, float* out_min, float* out_max)
{
  return SdfFromCellsHost<kEmitFloat>(cells, cell_bytes, nx, ny, nz, resolution,
                                      unknown_is_filled, add_virtual_border, object_ids,
                                      num_object_ids, false, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_from_cells_f64(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* sdf_out, double* out_min, double* out_max)
{
  return SdfFromCellsHost<kEmitDouble>(cells, cell_bytes, nx, ny, nz, resolution,
                                       unknown_is_filled, add_virtual_border, object_ids,
                                       num_object_ids, false, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_per_object_f32(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* sdf_out, float* out_min, float* out_max)
{
  return SdfFromCellsHost<kEmitFloat>(cells, cell_bytes, nx, ny, nz, resolution,
                                      unknown_is_filled, add_virtual_border, object_ids,
                                      num_object_ids, true, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_per_object_f64(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* sdf_out, double* out_min, double* out_max)
{
  return SdfFromCellsHost<kEmitDouble>(cells, cell_bytes, nx, ny, nz, resolution,
                                       unknown_is_filled, add_virtual_border, object_ids,
                                       num_object_ids, true, device, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_free_and_named_f32(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* sdf_out, float* out_min,
    float* out_max)
{
  return SdfFreeAndNamedHost<kEmitFloat>(cells, cell_bytes, nx, ny, nz, resolution,
                                         unknown_is_filled, add_virtual_border, device, sdf_out,
                                         out_min, out_max);
}

int vgt_b200_sdf_free_and_named_f64(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* sdf_out, double* out_min,
    double* out_max)
{
  return SdfFreeAndNamedHost<kEmitDouble>(cells, cell_bytes, nx, ny, nz, resolution,
                                          unknown_is_filled, add_virtual_border, device, sdf_out,
                                          out_min, out_max);
}

int vgt_b200_sdf_from_cells_f32_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max)
{
  return SdfCellsMultiDevice<kEmitFloat>(kCellSdf, cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, object_ids, num_object_ids,
                                     devices, num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_from_cells_f64_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max)
{
  return SdfCellsMultiDevice<kEmitDouble>(kCellSdf, cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, object_ids, num_object_ids,
                                     devices, num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_per_object_f32_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max)
{
  return SdfCellsMultiDevice<kEmitFloat>(kCellPerObject, cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, object_ids, num_object_ids,
                                     devices, num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_per_object_f64_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max)
{
  return SdfCellsMultiDevice<kEmitDouble>(kCellPerObject, cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, object_ids, num_object_ids,
                                     devices, num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_free_and_named_f32_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    float* sdf_out, float* out_min, float* out_max)
{
  return SdfCellsMultiDevice<kEmitFloat>(kCellFreeAndNamed, cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, nullptr, 0,
                                     devices, num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_free_and_named_f64_multi(
    const void* cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const int* devices, int num_devices,
    double* sdf_out, double* out_min, double* out_max)
{
  return SdfCellsMultiDevice<kEmitDouble>(kCellFreeAndNamed, cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, nullptr, 0,
                                     devices, num_devices, sdf_out, out_min, out_max);
}

int vgt_b200_sdf_from_cells_f32_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* d_sdf_out, float* d_min_max, void* stream)
{
  return SdfFromCellsDev<kEmitFloat>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, object_ids,
                                     num_object_ids, device, d_sdf_out, d_min_max,
                                     static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_from_cells_f64_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* d_sdf_out, double* d_min_max, void* stream)
{
  return SdfFromCellsDev<kEmitDouble>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                      unknown_is_filled, add_virtual_border, object_ids,
                                      num_object_ids, device, d_sdf_out, d_min_max,
                                      static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_per_object_f32_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, float* d_sdf_out, float* d_min_max, void* stream)
{
  return SdfPerObjectDev<kEmitFloat>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                     unknown_is_filled, add_virtual_border, object_ids,
                                     num_object_ids, device, d_sdf_out, d_min_max,
                                     static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_per_object_f64_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, const uint32_t* object_ids,
    int64_t num_object_ids, int device, double* d_sdf_out, double* d_min_max, void* stream)
{
  return SdfPerObjectDev<kEmitDouble>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                      unknown_is_filled, add_virtual_border, object_ids,
                                      num_object_ids, device, d_sdf_out, d_min_max,
                                      static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_free_and_named_f32_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, float* d_sdf_out,
    float* d_min_max, void* stream)
{
  return SdfFreeAndNamedDev<kEmitFloat>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                        unknown_is_filled, add_virtual_border, device, d_sdf_out,
                                        d_min_max, static_cast<cudaStream_t>(stream));
}

int vgt_b200_sdf_free_and_named_f64_dev(
    const void* d_cells, int cell_bytes, int64_t nx, int64_t ny, int64_t nz, double resolution,
    int unknown_is_filled, int add_virtual_border, int device, double* d_sdf_out,
    double* d_min_max, void* stream)
{
  return SdfFreeAndNamedDev<kEmitDouble>(d_cells, cell_bytes, nx, ny, nz, resolution,
                                         unknown_is_filled, add_virtual_border, device, d_sdf_out,
                                         d_min_max, static_cast<cudaStream_t>(stream));
}

int vgt_b200_edt_transform_inplace_f64(double* field, int64_t nx, int64_t ny, int64_t nz,
                                       int device)
{
  const int check = CheckSdfArguments(field, field, nx, ny, nz, 1.0);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (nz > 65535 * 32LL || ny > 65535 * 32LL || nx > 65535)
  {
    return FailInvalid("grid too large for the transpose launch");
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  KeepPoolMemory(device);
  return TransformFieldInPlace(field, nx, ny, nz);
}

void vgt_b200_reload_tuning(void)
{
  g_tuning.store(LoadTuning(), std::memory_order_release);
}

int vgt_b200_edt_sq_i32(
    const float* occupancy, int64_t nx, int64_t ny, int64_t nz, int unknown_is_filled, int device,
    int32_t* dist_to_filled_sq, int32_t* dist_to_free_sq)
{
  const int check = CheckSdfArguments(occupancy, dist_to_filled_sq, nx, ny, nz, 1.0);
  if (check != VGT_B200_OK)
  {
    return check;
  }
  if (dist_to_free_sq == nullptr)
  {
    return FailInvalid("null output pointer");
  }
  ScopedDevice scoped(device);
  VGT_CUDA_TRY(scoped.Status(), "cudaSetDevice");
  const int64_t count = nx * ny * nz;
  DeviceBuffer<float> d_in;
  DeviceBuffer<uint32_t> d_a;
  DeviceBuffer<uint32_t> d_b;
  DeviceBuffer<int32_t> d_filled;
  DeviceBuffer<int32_t> d_free;
  VGT_CUDA_TRY(d_in.Allocate(count), "cudaMalloc occupancy");
  VGT_CUDA_TRY(d_a.Allocate(count), "cudaMalloc packed field");
  VGT_CUDA_TRY(d_b.Allocate(count), "cudaMalloc packed field");
  VGT_CUDA_TRY(d_filled.Allocate(count), "cudaMalloc field");
  VGT_CUDA_TRY(d_free.Allocate(count), "cudaMalloc field");
  VGT_CUDA_TRY(cudaMemcpy(d_in.get(), occupancy, sizeof(float) * count, cudaMemcpyHostToDevice),
               "copy occupancy to device");
  int status = RunLocalPasses<float>(d_in.get(), nx, ny, nz, unknown_is_filled, d_a.get(),
                                     d_b.get(), nullptr);
  if (status != VGT_B200_OK)
  {
    return status;
  }
  uint32_t* d_packed = d_a.get();
  if (nx > 1)
  {
    status = LaunchEnvelope<kEmitPacked>(d_a.get(), d_b.get(), FamilyAlongX(nx, ny, nz),
                                         Square(nz - 1) + Square(ny - 1), FinalizeParams{},
                                         nullptr, nullptr);
    if (status != VGT_B200_OK)
    {
      return status;
    }
    d_packed = d_b.get();
  }
  const int threads = 256;
  SplitFieldsKernel<<<static_cast<unsigned>((count + threads - 1) / threads), threads>>>(
      d_packed, count, d_filled.get(), d_free.get()); NoteKernelLaunch();
  VGT_CUDA_TRY(cudaGetLastError(), "SplitFieldsKernel launch");
  VGT_CUDA_TRY(cudaMemcpy(dist_to_filled_sq, d_filled.get(), sizeof(int32_t) * count,
                          cudaMemcpyDeviceToHost),
               "copy field to host");
  VGT_CUDA_TRY(cudaMemcpy(dist_to_free_sq, d_free.get(), sizeof(int32_t) * count,
                          cudaMemcpyDeviceToHost),
               "copy field to host");
  return VGT_B200_OK;
}
}  // extern "C"
