// iqbb_kernels.cuh -- launch parameter blocks and launch wrappers of the IQBaseBand kernels.
#pragma once
#include "common.cuh"

namespace sdrg {

constexpr int kIqbbThreads = 256;      // threads per CTA of the accumulate kernels
constexpr int kIqbbPerThread = 8;      // consecutive FIR outputs per thread (register blocking)
constexpr int kIqbbTile = kIqbbThreads * kIqbbPerThread;   // input samples per CTA

// One process() call of the direct (unfolded) kernels.  All indices are relative to the first
// sample of the call; the host carries the global position (closed form, SURVEY.md 8 a1/a2).
struct IqbbAccumArgs {
  const void *x;          // n input samples (char2 / short2 / float2), device
  const void *hist_in;    // the previous `hist_len` samples (same type), device
  void       *hist_out;   // receives the last `hist_len` samples of [hist_in | x]
  const void *taps;       // int: Lp x int4 (Gauss form, see iqbb_kernels.cu); float: Lp float2
  const void *host_taps;  // the same int4 taps in host memory (enables the fixed-tap-count kernels), or null
  const void *lut;        // 128 x int2 or 128 x float2
  void       *acc_cur;    // window accumulators of this call (int2 / float2), slot 0 = open window
  void       *acc_next;   // accumulators of the next call: zeroed here (first `zero_next` entries)
  uint32_t    n;
  uint32_t    taps_len;   // Lp: number of (stripped) taps
  uint32_t    hist_len;   // Lp - 1
  uint32_t    ss;
  uint32_t    r0;         // position of sample 0 inside its window
  uint32_t    first;      // 1 if sample 0 is the very first sample since config() (window 0 has ss+1)
  uint32_t    phase0;     // NCO phase (15 bit) at sample 0
  uint32_t    inc;        // NCO increment mod 32768
  uint32_t    nco;        // 0: lut_inc == 0, the mixer is bypassed entirely (freqshift.hh:61)
  uint32_t    neg;        // negative frequency shift: idx = 127 - idx
  uint32_t    zero_next;
  uint32_t    in_fmt;     // int16 path only: 0 = complex<int16_t> input, 2 = complex uint8, 3 = complex int8 (fused AutoCast),
                          // 4 = REAL int16 (BaseBand<int16_t>, src/baseband.hh:304): sample = (x, 0);
                          // int8 path: 5 = REAL int8 (BaseBand<int8_t>): sample = (x, 0), FIR sum wrapped to 16 bits before the shift
  uint32_t    fir_shift;  // integer paths: the FIR result is shifted right by this (14 IQBaseBand, 16 BaseBand)
  uint32_t    div_m, div_s; // per-warp kernel: q / ss == (q * div_m) >> div_s for q < 2^31 (filled in by its launcher)
  uint32_t    zero;       // always 0: a third addend that keeps the kernel's plain additions on the ALU pipe (IADD3) --
                          // ptxas otherwise emits them as IMAD.IADD on the multiplier pipe, which is the one that is full
};

// One process() call of the folded float kernel (iqbb_fold_kernels.cu)
struct IqbbFoldArgs {
  const void   *x;          // n float2 samples
  void         *acc_cur;    // float2 window accumulators; slots n_out and n_out+1 stay open
  void         *acc_next;
  const float2 *tab_a;      // A(a), 128 entries
  const float2 *tab_u;      // U(r,e), 256 rows of taps_len entries
  uint32_t      n;
  uint32_t      taps_len;   // L
  uint32_t      ss;
  uint32_t      r0, first;
  uint32_t      phase0, inc;
  uint32_t      zero_next;
  // work decomposition, filled in by launch_iqbb_fold()
  uint32_t      part;       // a window longer than this is cut into pieces (chunks)
  uint32_t      cpw;        // chunks per window
  uint32_t      n_chunks;   // windows touched by this call x cpw
  uint32_t      chunks_per_warp;
  uint32_t      pf_dist;    // L2 prefetch distance in chunks of the same warp (0 = off)
  uint32_t      seg;        // TMA variant: samples per warp segment (multiple of 256)
  uint32_t      variant;    // 0/1 LDG loads (default), 2 TMA bulk-copy staging (needs 16-byte aligned input)
  // specialised schedule of a complete interior window (cpw == 1, taps_len <= 65), see iqbb_fold_f32_kernel
  uint32_t      fast;       // 1 = use it
  uint32_t      fast_nb;    // full 256-sample batches per window (ss / 256)
  uint32_t      fast_rs;    // 32-sample steps of the ragged batch (0..8)
  uint32_t      fast_pl;    // lanes of its last step (1..32)
  uint32_t      fast_hi;    // chunk ids 1..fast_hi are complete interior windows (0 = none)
  uint32_t     *work;       // window-pipelined kernel: work counter (0 at launch; the finalize kernel resets it)
  uint32_t      work_chunk; // consecutive windows per grab
  // per-window kernel (short windows), see iqbb_fold_perwin.cu: V(class, j), one row per distinct carry pattern
  const float2 *tab_v;      // v_rows x v_pitch, or null when the table is not built (window too long / table too large)
  const uint16_t *tab_cls;  // 256 entries: low phase byte at a window's first sample -> row of tab_v
  uint32_t      v_rows, v_pitch;
  uint32_t      d_lo, d_hi; // slots d_lo..d_hi are complete windows whose L-1 halo samples lie inside this call (filled in by the launcher)
};

// finalize (+ optional demodulation) of the completed windows of one call
struct IqbbFinalizeArgs {
  uint32_t   *work_reset; // accumulate kernel's work counter, set back to 0 here (may be null)
  const void *acc_cur;    // n_out completed slots followed by the open one
  void       *acc_next;   // slots 0 and 1 receive the carry (open window, and the one after it)
  void       *bb_out;     // complex Scalar[n_out] or null
  void       *audio_out;  // demod output or null
  const void *fm_last_in; // carried FM angle (int16 as int32 / double), device scalar
  void       *fm_last_out;
  uint32_t    n_out;
  uint32_t    ss;
  uint32_t    demod;      // SDRG_DEMOD_*
  uint32_t    e0;         // call-relative index of the sample that completes slot 0
  uint64_t    seg;        // buffer_size (segment length in input samples); 0 = one segment
  uint32_t    in_place;   // FM: what element 0 of every segment shows
  uint32_t    narrow16;   // BaseBand<int8_t>: the window sum and the division run in int16 (complex<int16_t>::operator/=)
};

// One process() call of a channel bank (bank_kernels.cu); window geometry as in IqbbAccumArgs
struct BankAccumArgs {
  const void     *x, *hist_in;
  void           *hist_out;
  const void     *taps;       // int: channels x taps_len int4 (Gauss form); float: taps_len x (channels rounded up to 32) float2
  const void     *lut;        // 128 x int2 / float2 (shared by all channels)
  const void     *tab_u;      // float: U_c(r, 0) per group of 32 channels, [group][r][channel in group] float2
  const uint32_t *inc;        // per channel: lut_inc (0 = mixer bypassed)
  const uint32_t *neg;        // per channel: negative shift
  void           *acc_cur, *acc_next;   // channels x acc_stride accumulators (int2)
  size_t          acc_stride;
  uint32_t        n, channels, group, taps_len, hist_len, ss, r0, first;
  uint32_t        consumed15; // samples consumed since config(), mod 32768 (NCO phase = consumed*inc mod 32768)
  uint32_t        zero_next;
};
struct BankFinalizeStrides { size_t acc_stride, out_stride; uint32_t bb_bytes, audio_bytes; };

int launch_iqbb_accum(int scalar, const IqbbAccumArgs &a, cudaStream_t st);
int launch_bank_accum(int scalar, const BankAccumArgs &a, cudaStream_t st);
int launch_bank_finalize(int scalar, const IqbbFinalizeArgs &a, const BankFinalizeStrides &s, uint32_t channels, cudaStream_t st);
int launch_iqbb_finalize(int scalar, const IqbbFinalizeArgs &a, cudaStream_t st);
int launch_iqbb_fold(const IqbbFoldArgs &a, cudaStream_t st, int *which = nullptr);   // *which: see sdrg_iqbb_last_float_kernel

// stand-alone demodulators (demod_kernels.cu)
int launch_fmdemod(int scalar, const void *in, size_t n, void *out, const void *last_in, void *last_out,
                   int in_place, cudaStream_t st);
int launch_amdemod(int scalar, const void *in, size_t n, void *out, cudaStream_t st);
int launch_usbdemod(int scalar, const void *in, size_t n, void *out, cudaStream_t st);
// AutoCast<complex<int16_t>> from complex uint8 (fmt 2) / int8 (fmt 3): n_bytes in, n_bytes int16 out
int launch_autocast_cs16(int fmt, const void *in, size_t n_bytes, void *out, cudaStream_t st);
// the whole AutoCast table: kind 1..14 (demod_kernels.cu), n_scalars input scalars
int launch_autocast(int kind, const void *in, size_t n_scalars, void *out, cudaStream_t st);
// FMDeemph<int16_t>: `streams` independent sequences of n samples (stride elements apart), one thread each
int launch_fmdeemph(const void *in, void *out, size_t n, size_t streams, size_t stride, int alpha, void *avg, cudaStream_t st);

}  // namespace sdrg
