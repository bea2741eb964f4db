/* sdrg.h -- C ABI of the B200-native libsdr receive-chain hot path.
 *
 * This is the drop-in boundary: a plain-C shared library (libsdrg.so) whose entry points are what
 * libsdr's node classes bind to.  Each group cites the reference interface it replaces
 * (file:line relative to the libsdr source tree).  The C++ node classes that keep libsdr's
 * sdr::Sink<T>/Source/Buffer<T> config()/process() surface on top of these calls live in
 * include/sdrg/ (see INTEGRATION.md).
 *
 * Conventions
 *  - every call returns an sdrg status (0 = ok); sdrg_last_error() gives the thread-local message.
 *    SDRG_ERR_CONFIG maps to sdr::ConfigError, everything else to sdr::RuntimeError
 *    (src/exception.hh:10-45).
 *  - "_dev" entry points take DEVICE pointers and a cudaStream_t (passed as void*) and are
 *    asynchronous; the others take HOST pointers, include the host<->device copies and return
 *    after the result is in host memory.
 *  - IQ samples are interleaved (re, im) pairs exactly like std::complex<T> arrays.
 *  - there is no CPU fallback: without a CUDA device every compute call fails with SDRG_ERR_CUDA.
 */
#ifndef SDRG_H
#define SDRG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDRG_ABI_VERSION 2

enum {
  SDRG_OK = 0,
  SDRG_ERR_CONFIG = 1,   /* -> sdr::ConfigError  */
  SDRG_ERR_RUNTIME = 2,  /* -> sdr::RuntimeError */
  SDRG_ERR_CUDA = 3,     /* -> sdr::RuntimeError */
  SDRG_ERR_ARG = 4       /* -> sdr::RuntimeError */
};

/* sdr::Config::Type (src/node.hh:39-53), same numeric values. */
enum {
  SDRG_T_UNDEFINED = 0, SDRG_T_U8, SDRG_T_S8, SDRG_T_U16, SDRG_T_S16, SDRG_T_F32, SDRG_T_F64,
  SDRG_T_CU8, SDRG_T_CS8, SDRG_T_CU16, SDRG_T_CS16, SDRG_T_CF32, SDRG_T_CF64
};

/* sdr::Config (src/node.hh:35-105). */
typedef struct {
  int    type;
  double sample_rate;
  size_t buffer_size;
  size_t num_buffers;
} sdrg_config;

/* ---- runtime ---------------------------------------------------------------------------------- */
int         sdrg_abi_version(void);
/* Always 0: the library is built one way only, and no environment variable can change what it computes or which
 * kernel it launches.  Kept so that existing callers of this check keep working.  Returns the flag itself, not a
 * status. */
int         sdrg_build_has_experiments(void);
const char *sdrg_last_error(void);
int         sdrg_device_count(int *count);
int         sdrg_set_device(int device);          /* device used by handles created afterwards on this thread */
int         sdrg_get_device(int *device);         /* the calling thread's device (threads start on device 0) */
int         sdrg_device_synchronize(void);

/* ---- buffer storage (replaces the malloc in RawBuffer::RawBuffer(size_t, BufferOwner*),
 *      src/buffer.cc:23-33): pinned host memory with a same-sized device mirror.  The device-valid
 *      range records what a GPU node last produced, so that chained GPU nodes skip the round trip
 *      and host-only sinks get a copy back on demand. ------------------------------------------- */
int sdrg_buffer_alloc(size_t bytes, void **host_ptr);
int sdrg_buffer_free(void *host_ptr);
int sdrg_buffer_is_managed(const void *host_ptr, int *managed);
int sdrg_buffer_device_ptr(const void *host_ptr, void **dev_ptr);            /* host_ptr may point inside an allocation */
int sdrg_buffer_mark_device_valid(const void *host_ptr, size_t bytes, void *stream); /* [host_ptr, +bytes) now lives on the device */
int sdrg_buffer_device_valid(const void *host_ptr, size_t bytes, int *valid);
int sdrg_buffer_invalidate_device(const void *host_ptr);                     /* host becomes authoritative again */
int sdrg_buffer_sync_to_host(const void *host_ptr, size_t bytes);            /* no-op unless the range is device-valid and unsynced */
/* Device address of [host_ptr, +bytes) with the data present: a device-valid range is used as is,
 * anything else is copied up first (async on `stream`; pinned, so truly asynchronous).  For memory
 * that is NOT a managed buffer, *dev_ptr is set to NULL and the caller stages it itself. */
int sdrg_buffer_to_device(const void *host_ptr, size_t bytes, void *stream, void **dev_ptr);

/* The library's compute stream (one per device, non-blocking): nodes that chain on the device
 * launch on it so that producer -> consumer order needs no events. */
int sdrg_stream_default(void **stream);
int sdrg_stream_synchronize(void *stream);
/* device scratch of at least `bytes`, private to the calling thread, valid until its next call */
int sdrg_scratch(size_t bytes, void **dev_ptr);
/* a second such scratch, for results that are copied back to foreign (unmanaged) host memory while an input
 * staged in the first one is still being read */
int sdrg_scratch_out(size_t bytes, void **dev_ptr);
int sdrg_memcpy_h2d_async(void *d_dst, const void *h_src, size_t bytes, void *stream);
int sdrg_memcpy_d2h_async(void *h_dst, const void *d_src, size_t bytes, void *stream);

/* ---- IQBaseBand<Scalar> (src/baseband.hh:21-297; FreqShiftBase src/freqshift.hh:13-107) -------
 * scalar: SDRG_T_S8, SDRG_T_S16 or SDRG_T_F32.  Integer paths are bit-exact w.r.t. the reference;
 * the float path is defined in DESIGN.md (the reference does not compile for float). */
typedef struct sdrg_iqbb sdrg_iqbb;

int sdrg_iqbb_create(int scalar, double Fc, double Ff, double width, size_t order,
                     size_t sub_sample, double oFs, sdrg_iqbb **h);   /* ctor, baseband.hh:47-57 */
/* Real-input BaseBand<int16_t>(Fc, Ff, width, order, sub_sample) (src/baseband.hh:304-529): the same
 * handle type and process calls, input elements are REAL int16 samples (SDRG_T_S16, 2 bytes each), output
 * complex int16.  FIR gain 2^16, windows of exactly sub_sample samples, rates kept in double. */
int sdrg_iqbb_create_real(int scalar, double Fc, double Ff, double width, size_t order,
                          size_t sub_sample, sdrg_iqbb **h);           /* ctor, baseband.hh:339-350 */
int sdrg_iqbb_destroy(sdrg_iqbb *h);
int sdrg_iqbb_set_center_frequency(sdrg_iqbb *h, double Fc);          /* baseband.hh:84-86  */
int sdrg_iqbb_set_filter_frequency(sdrg_iqbb *h, double Ff);          /* baseband.hh:91-93  */
int sdrg_iqbb_set_filter_width(sdrg_iqbb *h, double width);           /* baseband.hh:98-100 */
int sdrg_iqbb_set_order(sdrg_iqbb *h, size_t order);                  /* baseband.hh:69-79 (history is zeroed, see DESIGN.md) */
int sdrg_iqbb_set_subsample(sdrg_iqbb *h, size_t sub_sample);         /* baseband.hh:105-107 */
int sdrg_iqbb_set_output_sample_rate(sdrg_iqbb *h, double oFs);       /* baseband.hh:110-112 */
/* config(): SDRG_ERR_CONFIG on a type mismatch; a config without type/rate/buffer size is ignored
 * (returns SDRG_OK with out->type == SDRG_T_UNDEFINED).  Resets the stream state. baseband.hh:115-194 */
int sdrg_iqbb_configure(sdrg_iqbb *h, const sdrg_config *src, sdrg_config *out);
/* The host half of config() only (type check, sub-sampling, kernel, LUT increment, output config):
 * touches no device, leaves the handle unconfigured for process().  Lets the design be inspected
 * (sdrg_iqbb_get_info) on a machine without a GPU. */
int sdrg_iqbb_design(sdrg_iqbb *h, const sdrg_config *src, sdrg_config *out);

/* AutoCast fused into the load (examples/sdr_fm.cc:39,49-50 put AutoCast< complex<int16_t> > in front
 * of IQBaseBand<int16_t>): with type SDRG_T_CU8 or SDRG_T_CS8 an int16 node consumes the raw complex
 * 8-bit stream and converts on the fly exactly like src/autocast.hh:187-204 (2 bytes per sample from
 * HBM instead of 4, no separate pass).  Call before config(); config() then expects that type. */
int sdrg_iqbb_set_input_type(sdrg_iqbb *h, int type);

/* SDRG_T_F32 only: which accumulate kernel config() selects.  0 = auto (folded when
 * sub_sample >= max(2, order-1), else direct), 1 = direct (sample-by-sample FIR, FMA-bound),
 * 2 = folded (one weight per input sample, HBM-bound; SDRG_ERR_CONFIG at config() if not eligible).
 * 3 (formerly folded with TMA bulk-copy staging) is refused with SDRG_ERR_CONFIG.
 * Must be called before config(). */
int sdrg_iqbb_set_float_path(sdrg_iqbb *h, int mode);

/* Diagnostics (no reference counterpart): which accumulate kernel the node's last process() call launched.
 * 0 = none yet / integer node, 1 = direct FIR, 2 = folded (batched, any window length), 3 = folded, window-pipelined
 * (sub_sample <= 512), 4 = folded, staged short windows, 5 = folded, one thread group per window
 * (iqbb_fold_perwin.cu).  6 (formerly folded, TMA staging) is no longer returned. */
int sdrg_iqbb_last_float_kernel(const sdrg_iqbb *h, int *which);

/* What config() derived; kernel/lut are written only when non-NULL (order / 128 int32 pairs, resp.
 * float pairs for SDRG_T_F32). */
typedef struct {
  size_t   order;
  size_t   sub_sample;
  size_t   lut_inc;
  int      negative_shift;
  uint64_t samples_consumed;
  uint64_t outputs_produced;
} sdrg_iqbb_info;
int sdrg_iqbb_get_info(const sdrg_iqbb *h, sdrg_iqbb_info *info, void *kernel, void *lut);

/* process(): n_in complex samples in, the completed averages out (baseband.hh:136-223).
 * *n_out is computed on the host (closed form) and is valid on return from both variants. */
int sdrg_iqbb_process(sdrg_iqbb *h, const void *in, size_t n_in, void *out, size_t out_cap, size_t *n_out);
int sdrg_iqbb_process_dev(sdrg_iqbb *h, const void *d_in, size_t n_in, void *d_out, size_t out_cap,
                          size_t *n_out, void *stream);
/* number of outputs the next process() of n_in samples will deliver */
int sdrg_iqbb_outputs_for(const sdrg_iqbb *h, size_t n_in, size_t *n_out);

/* ---- demodulators (src/demod.hh) -------------------------------------------------------------- */
enum { SDRG_DEMOD_NONE = 0, SDRG_DEMOD_FM = 1, SDRG_DEMOD_AM = 2, SDRG_DEMOD_USB = 3 };

/* FMDemod<iScalar,oScalar> (demod.hh:172-266, fast_atan2 src/math.hh:9-40).
 * in_scalar S8/S16 -> int16 output; F32 -> float output (defined in DESIGN.md).
 * Element 0 of every processed buffer is skipped exactly like the reference: with in_place != 0 it
 * shows the bytes of the input that alias it, otherwise the output element is left untouched.
 * The _dev variants accept d_out == d_in (true in-place use, demod.hh:233-234): the result is then
 * formed in scratch memory and copied over the input in stream order. */
typedef struct sdrg_fmdemod sdrg_fmdemod;
int sdrg_fmdemod_create(int in_scalar, sdrg_fmdemod **h);
int sdrg_fmdemod_destroy(sdrg_fmdemod *h);
int sdrg_fmdemod_configure(sdrg_fmdemod *h, const sdrg_config *src, sdrg_config *out);  /* demod.hh:195-226 */
int sdrg_fmdemod_process(sdrg_fmdemod *h, const void *in, size_t n, void *out, int in_place);
int sdrg_fmdemod_process_dev(sdrg_fmdemod *h, const void *d_in, size_t n, void *d_out, int in_place, void *stream);

/* AMDemod<Scalar> (demod.hh:16-86) and USBDemod<Scalar> (demod.hh:91-166): stateless. */
int sdrg_amdemod_configure(int scalar, const sdrg_config *src, sdrg_config *out);       /* demod.hh:35-62 */
int sdrg_usbdemod_configure(int scalar, const sdrg_config *src, sdrg_config *out);      /* demod.hh:117-142 */
int sdrg_amdemod_process(int scalar, const void *in, size_t n, void *out);
int sdrg_amdemod_process_dev(int scalar, const void *d_in, size_t n, void *d_out, void *stream);
int sdrg_usbdemod_process(int scalar, const void *in, size_t n, void *out);
int sdrg_usbdemod_process_dev(int scalar, const void *d_in, size_t n, void *d_out, void *stream);

/* ---- the nodes either side of the path (SURVEY.md 8f) ------------------------------------------
 * AutoCast<Scalar> (src/autocast.hh:13-262), the whole table of :30-69: out_type S8 / CS8 / S16 / CS16 from
 * u8 / s8 / u16 / s16 and, for the complex outputs, cu8 / cs8 / cu16 / cs16; `n` counts input ELEMENTS of in_type
 * (a complex sample is one element).  Every cast reproduces the reference's arithmetic including its quirks (cu8 read
 * through int8_t*, the constants (2<<15)-1 and 1<<15).  A pair the reference refuses is SDRG_ERR_CONFIG with its message. */
int sdrg_autocast_out_bytes(int in_type, int out_type, size_t n, size_t *bytes);   /* bytes n input elements turn into */
int sdrg_autocast_process(int in_type, int out_type, const void *in, size_t n, void *out);
int sdrg_autocast_process_dev(int in_type, int out_type, const void *d_in, size_t n, void *d_out, void *stream);
/* FMDeemph<int16_t> (src/demod.hh:271-362): integer 1-pole IIR with rounding.  `streams` independent
 * sequences (e.g. the channels of a bank), each n samples long, `stride` elements apart; the running
 * average of every stream is carried across calls and reset by configure(). */
typedef struct sdrg_fmdeemph sdrg_fmdeemph;
int sdrg_fmdeemph_create(size_t streams, sdrg_fmdeemph **h);
int sdrg_fmdeemph_destroy(sdrg_fmdeemph *h);
int sdrg_fmdeemph_configure(sdrg_fmdeemph *h, const sdrg_config *src, sdrg_config *out);
int sdrg_fmdeemph_process(sdrg_fmdeemph *h, const void *in, size_t n, size_t stride, void *out);
int sdrg_fmdeemph_process_dev(sdrg_fmdeemph *h, const void *d_in, size_t n, size_t stride, void *d_out, void *stream);

/* ---- receive chain: IQBaseBand -> demod, many buffers per launch ------------------------------
 * Equivalent to n_buffers consecutive Source::send() calls of buffer_size samples each through
 * IQBaseBand<Scalar> -> {FM,AM,USB}Demod connected directly and in place (examples/sdr_fm.cc:48-51,
 * src/node.cc:66-84): one fused pass on the device, intermediate base-band samples never leave
 * HBM/L2.  Outputs are dense; counts[b] (host array, n_buffers entries, may be NULL) receives the
 * number of outputs of buffer b.  d_bb / bb may be NULL when the base-band samples are not wanted. */
typedef struct sdrg_rxchain sdrg_rxchain;
int sdrg_rxchain_create(sdrg_iqbb *bb, int demod, sdrg_rxchain **h);   /* borrows bb; bb must outlive the chain */
int sdrg_rxchain_destroy(sdrg_rxchain *h);
int sdrg_rxchain_reset(sdrg_rxchain *h);                               /* demod state only (FM last value) */
int sdrg_rxchain_process_dev(sdrg_rxchain *h, const void *d_in, size_t buffer_size, size_t n_buffers,
                             void *d_bb, void *d_audio, size_t out_cap, size_t *n_out, size_t *counts,
                             void *stream);
int sdrg_rxchain_process(sdrg_rxchain *h, const void *in, size_t buffer_size, size_t n_buffers,
                         void *bb, void *audio, size_t out_cap, size_t *n_out, size_t *counts);
/* ---- FFTPlan<float> (src/fftplan.hh:11-34, src/fftplan_fftw3.hh:79-142; FFTW3 is replaced by
 *      hand-written FFT kernels).  Unnormalised c2c DFT, direction 0 = FORWARD (exp(-i..)),
 *      1 = BACKWARD.  ANY size 1..2^24 like the reference's FFTW plan (fftplan_fftw3.hh:83-106):
 *      powers of two up to 8192 run in shared memory (the hot sizes), larger powers of two as a
 *      four-step decomposition, every other size through Bluestein's convolution.  An empty buffer is
 *      SDRG_ERR_CONFIG (fftplan_fftw3.hh:87-97).  `batch` transforms are contiguous. ---------------- */
typedef struct sdrg_fft sdrg_fft;
int sdrg_fft_create(size_t n, int direction, sdrg_fft **h);
int sdrg_fft_destroy(sdrg_fft *h);
int sdrg_fft_exec(sdrg_fft *h, const void *in, void *out, size_t batch);
int sdrg_fft_exec_dev(sdrg_fft *h, const void *d_in, void *d_out, size_t batch, void *stream);
/* FFTPlan<double> (src/fftplan_fftw3.hh:12-75): complex double, any size 1..2^22, double arithmetic on the device
 * (radix-2 passes through global memory, Bluestein for sizes that are not a power of two; not a hot path). */
typedef struct sdrg_fft64 sdrg_fft64;
int sdrg_fft64_create(size_t n, int direction, sdrg_fft64 **h);
int sdrg_fft64_destroy(sdrg_fft64 *h);
int sdrg_fft64_exec(sdrg_fft64 *h, const void *in, void *out, size_t batch);
int sdrg_fft64_exec_dev(sdrg_fft64 *h, const void *d_in, void *d_out, size_t batch, void *stream);

/* ---- FilterNode<float> (src/filternode.hh:231-283): FilterSink (forward FFT of 2*block, shared) +
 *      one FilterSource per added filter (spectrum multiply, backward FFT, overlap), and the
 *      BufferNode that re-chunks arbitrary input sizes to `block` samples (src/buffernode.hh).
 *      Complex float in, complex float out; ANY block size 1..2^22 (filternode.hh:236): powers of two
 *      up to 4096 run the fused overlap-save kernels, other sizes a gather / batched-FFT / crop
 *      composition with FFT size 2^ceil(log2 2 block) -- same taps, same normalisation, same result. */
typedef struct sdrg_filter sdrg_filter;
int sdrg_filter_create(size_t block_size, sdrg_filter **h);                      /* filternode.hh:236-246 */
int sdrg_filter_destroy(sdrg_filter *h);
int sdrg_filter_add(sdrg_filter *h, double fmin, double fmax, size_t *index);    /* addFilter, filternode.hh:262-270 */
int sdrg_filter_set_freq(sdrg_filter *h, size_t index, double fmin, double fmax);/* FilterSource::setFreq, :128-130 */
int sdrg_filter_count(const sdrg_filter *h, size_t *n);
int sdrg_filter_configure(sdrg_filter *h, const sdrg_config *src, sdrg_config *out);   /* filternode.hh:56-79,133-160 */
/* kern: 2*block complex floats (normalised spectrum), taps: block complex floats; either may be NULL */
int sdrg_filter_get_design(const sdrg_filter *h, size_t index, void *kern_2n, void *taps_n);
int sdrg_filter_outputs_for(const sdrg_filter *h, size_t n_in, size_t *n_out);
/* filter f's output lands at out + f*out_stride (in samples); *n_out = samples produced per filter */
int sdrg_filter_process(sdrg_filter *h, const void *in, size_t n_in, void *out, size_t out_stride, size_t *n_out);
int sdrg_filter_process_dev(sdrg_filter *h, const void *d_in, size_t n_in, void *d_out, size_t out_stride,
                            size_t *n_out, void *stream);

/* ---- channel bank: C independent IQBaseBand<Scalar> nodes on ONE input stream, each followed by
 *      FM / AM / USB demodulators connected out of place (several sinks on one source,
 *      src/node.cc:75).  Channel c equals IQBaseBand<Scalar>(Fc[c], Ff[c], width, order, sub_sample, oFs)
 *      (src/baseband.hh:47-57) bit for bit; Ff == NULL means Ff = Fc.  scalar: SDRG_T_S8 / SDRG_T_S16, or
 *      SDRG_T_F32: input complex float, outputs as sdrg_rxchain's float chain (base band float2, FM / AM /
 *      USB float), each channel equal to the float node to float rounding; sdrg_bank_get_info then returns
 *      float taps (as sdrg_iqbb_get_info).  Every scalar needs sub_sample >= 256 and order <= 256.
 *      Outputs of channel c land at <ptr> + c*out_stride elements; any output pointer may be NULL. -- */
typedef struct sdrg_bank sdrg_bank;
int sdrg_bank_create(int scalar, size_t n_channels, const double *Fc, const double *Ff, double width, size_t order,
                     size_t sub_sample, double oFs, sdrg_bank **h);
int sdrg_bank_destroy(sdrg_bank *h);
int sdrg_bank_configure(sdrg_bank *h, const sdrg_config *src, sdrg_config *out);
int sdrg_bank_get_info(const sdrg_bank *h, size_t *channels, size_t *sub_sample, size_t channel, sdrg_iqbb_info *info, void *kernel);
int sdrg_bank_outputs_for(const sdrg_bank *h, size_t n_in, size_t *n_out);
int sdrg_bank_process(sdrg_bank *h, const void *in, size_t buffer_size, size_t n_buffers, void *bb, void *fm, void *am,
                      void *usb, size_t out_stride, size_t *n_out);
int sdrg_bank_process_dev(sdrg_bank *h, const void *d_in, size_t buffer_size, size_t n_buffers, void *d_bb, void *d_fm,
                          void *d_am, void *d_usb, size_t out_stride, size_t *n_out, void *stream);

/* ---- multi-GPU (SURVEY.md 8e) -----------------------------------------------------------------------
 * The reference has no parallelism (its only thread is the Queue's, src/queue.cc:57-60); the path shards
 * over independent channels / streams and only demodulated outputs cross GPUs.  Both mechanisms below use
 * plain peer memory: output rows are written by the producing GPU's finalize kernel (or a copy engine)
 * directly into the consumer GPU's HBM over NVLink, so no collective kernel competes for SMs.
 *
 * (1) One process, G devices: a channel bank whose channels are sharded by contiguous ranges over
 *     `devices` (shard g owns channels [g*C/G, (g+1)*C/G), the first C%G shards one more).  Same
 *     semantics and bit-identical results as sdrg_bank_* with all channels on one device (int8, int16;
 *     SDRG_T_F32 is accepted too, each shard being a float bank, equal to it to float rounding).
 *     _process:     host pointers; every device uploads the input and returns its rows; blocking.
 *     _process_dev: input and output arrays live on devices[0]; `stream` is a stream of devices[0]; the
 *                   input is broadcast with copy-engine peer copies, shards with peer access store their
 *                   rows straight into the output arrays (others stage + peer copy); asynchronous, `stream`
 *                   is ordered behind all shards on return. */
typedef struct sdrg_bank_sharded sdrg_bank_sharded;
int sdrg_bank_sharded_create(int scalar, size_t n_channels, const double *Fc, const double *Ff, double width, size_t order,
                             size_t sub_sample, double oFs, const int *devices, size_t n_devices, sdrg_bank_sharded **h);
int sdrg_bank_sharded_destroy(sdrg_bank_sharded *h);
int sdrg_bank_sharded_configure(sdrg_bank_sharded *h, const sdrg_config *src, sdrg_config *out);
int sdrg_bank_sharded_info(const sdrg_bank_sharded *h, size_t *channels, size_t *n_shards, size_t shard, int *device,
                           size_t *first_channel, size_t *n_shard_channels, int *direct_peer_stores);
int sdrg_bank_sharded_outputs_for(const sdrg_bank_sharded *h, size_t n_in, size_t *n_out);
int sdrg_bank_sharded_process(sdrg_bank_sharded *h, const void *in, size_t buffer_size, size_t n_buffers, void *bb, void *fm,
                              void *am, void *usb, size_t out_stride, size_t *n_out);
int sdrg_bank_sharded_process_dev(sdrg_bank_sharded *h, const void *d_in, size_t buffer_size, size_t n_buffers, void *d_bb,
                                  void *d_fm, void *d_am, void *d_usb, size_t out_stride, size_t *n_out, void *stream);

/* (2) One process per GPU: peer windows.  The consumer creates a window in its HBM and ships the 64-byte
 *     handle to the producers (any host channel); a producer opens it and uses addresses inside it as
 *     output pointers of the *_process_dev calls.  sdrg_peer_signal() publishes a 64-bit progress value
 *     into a slot (stream-ordered after everything enqueued before it, system-scope release);
 *     sdrg_peer_wait() holds `stream` until all n_slots consecutive slots are >= value (or timeout_ms
 *     passed: sdrg_peer_wait_timed_out() then reports 1 once; 0 = 10 s).  Windows start zeroed. */
#define SDRG_IPC_HANDLE_BYTES 64
int sdrg_peer_window_create(size_t bytes, void **d_ptr, void *ipc_handle);
int sdrg_peer_window_open(const void *ipc_handle, void **d_ptr);
int sdrg_peer_window_close(void *d_ptr);
int sdrg_peer_window_destroy(void *d_ptr);
int sdrg_peer_signal(void *d_slot, uint64_t value, void *stream);
int sdrg_peer_wait(const void *d_slots, size_t n_slots, uint64_t value, unsigned timeout_ms, void *stream);
int sdrg_peer_wait_timed_out(int *timed_out);
int sdrg_memcpy_d2d_async(void *d_dst, const void *d_src, size_t bytes, void *stream);   /* same or peer device */
/* Pinned host memory for feeding `device`: bound to the NUMA node the GPU hangs off (sysfs numa_node; *numa_node
 * receives it, -1 = unknown / single node, then plain cudaHostAlloc).  For the host-pointer entry points. */
int sdrg_host_alloc(size_t bytes, int device, void **host_ptr, int *numa_node);
int sdrg_host_free(void *host_ptr);

/* number of kernels the library has launched so far (all handles, this process) */
int sdrg_kernel_launch_count(uint64_t *count);

/* ---- measurement hooks: CUDA events recorded on the launching stream around each kernel of the
 *      given kind while enabled; sdrg_profile_read() waits for them, returns the summed device
 *      time and the launch count, and clears them. ---------------------------------------------- */
enum { SDRG_KERNEL_IQBB_ACCUM = 1, SDRG_KERNEL_IQBB_FINALIZE = 2, SDRG_KERNEL_OLA = 3, SDRG_KERNEL_BANK = 4 };
int sdrg_profile_enable(int on);
int sdrg_profile_read(int kind, double *total_ms, uint64_t *launches);

#ifdef __cplusplus
}
#endif
#endif /* SDRG_H */
