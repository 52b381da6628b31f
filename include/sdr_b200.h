/* sdr_b200.h -- C ABI of the B200 IQ->PCM demodulation engine.
 *
 * The reference (wizardyesterday/RtlSdrDiags) has no FFI layer: its boundary for
 * this path is a set of C++ classes, one object per radio. This header is the
 * boundary a maintainer binds instead; one engine stands for a BANK of
 * n_channels independent radios on one GPU. Each entry point names the
 * reference interface it replaces.
 *
 *   reference (radioDiags/)                               this ABI
 *   ----------------------------------------------------  -------------------------
 *   new IqDataProcessor + new {Am,Fm,WbFm,Ssb}Demodulator  sdr_engine_create
 *     (src_diags/Radio.cc:150-181)
 *   IqDataProcessor::setDemodulatorMode                    sdr_set_mode / sdr_set_modes
 *     (src_diags/IqDataProcessor.cc:236-262)
 *   XDemodulator::setDemodulatorGain                       sdr_set_gain / sdr_set_gain_all
 *     (AmDemodulator.cc:267, FmDemodulator.cc:304,
 *      WbFmDemodulator.cc:341, SsbDemodulator.cc:390)
 *   XDemodulator::resetDemodulator                         sdr_reset
 *     (AmDemodulator.cc:232, FmDemodulator.cc:271,
 *      WbFmDemodulator.cc:304, SsbDemodulator.cc:297)
 *   IqDataProcessor::acceptIqData(ts, u8*, n)              sdr_accept_iq(.., SDR_IQ_U8_OFFSET)
 *     (src_diags/IqDataProcessor.cc:722-840)
 *   XDemodulator::acceptIqData(int8_t*, n)                 sdr_accept_iq(.., SDR_IQ_S8_ROTATED)
 *     (e.g. FmDemodulator.cc:334-352)
 *   pcmCallbackPtr(int16_t*, n)  (radioApp.cc:103-111)     sdr_get_pcm / sdr_pcm_device
 *   IqDataProcessor::setSignalDetectThreshold              sdr_set_squelch_threshold
 *     (src_diags/IqDataProcessor.cc:284-295)
 *   radio_adjustableReceiveGainInDb (IqDataProcessor.cc:8) sdr_set_receive_gain_db
 *   signal-state / signal-magnitude callbacks              sdr_enable_signal_reports,
 *     (src_diags/IqDataProcessor.cc:771-790)                sdr_get_signal
 *   IqDataProcessor::enableIqDump / disableIqDump          sdr_set_iq_dump
 *     (src_diags/IqDataProcessor.cc:633-669)
 *   networkInterfacePtr->sendData(signedBufferPtr, n)      sdr_get_iq_dump / sdr_iq_dump_device
 *     (IqDataProcessor.cc:756-760, UdpClient.cc:173-241)
 *   DataConsumer::acceptData(ts, buf, n) + consumer thread  sdr_ingest_accept / _acquire+_commit,
 *     (src_diags/DataConsumer.cc:220-261, 318-352)           sdr_ingest_retire, sdr_ingest_stats
 *   Radio's demodulator objects, one set per radio, and    sdr_bank_create, sdr_bank_set_mode(s),
 *     one DataConsumer feeding them (Radio.cc:150-187,       sdr_bank_acquire + sdr_bank_commit,
 *     DataConsumer.cc:220-352) -- for radios spread over     sdr_bank_retire
 *     several GPUs of one box
 *   new Decimator / Interpolator / Decimator_int16 /        sdr_filter_bank_create
 *     Interpolator_int16 (N, taps, factor)
 *     (Filters/Decimator.cc:41-76, Filters/Interpolator.cc:39-61, Filters/Int16/*.cc)
 *   decimate(x, &y) / interpolate(x, y[L]) per sample       sdr_filter_bank_run (blocks of samples)
 *     (Filters/Decimator.cc:281-322, Filters/Interpolator.cc interpolate)
 *   resetFilterState()                                      sdr_filter_bank_reset
 *   new IirFilter(nb, b, na, a)                             sdr_filter_bank_create_iir
 *     (Filters/IirFilter.cc, IirFilter.h)
 *   IirFilter::filterData(x) per sample                     sdr_filter_bank_run (blocks of samples)
 *   IirFilter::resetFilterState()                           sdr_filter_bank_reset
 *
 * All functions return 0 on success or a negative SDR_E_* code; none throws.
 * Calls on one engine must be serialised by the caller (the reference calls
 * acceptIqData from one thread, DataConsumer.cc:342). There is no CPU fallback:
 * without a usable CUDA device sdr_engine_create fails with SDR_E_CUDA.
 */
#ifndef SDR_B200_H
#define SDR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sdr_engine sdr_engine;

/* IqDataProcessor::demodulatorType, hdr_diags/IqDataProcessor.h:20 */
enum { SDR_MODE_NONE = 0, SDR_MODE_AM = 1, SDR_MODE_FM = 2, SDR_MODE_WBFM = 3,
       SDR_MODE_LSB = 4, SDR_MODE_USB = 5 };
/* which of a channel's four demodulator objects a gain / reset addresses */
enum { SDR_KIND_AM = 1, SDR_KIND_FM = 2, SDR_KIND_WBFM = 3, SDR_KIND_SSB = 4 };
/* FM/WBFM PCM scaling: radioDiags/ (gain/deviation*32767, FmDemodulator.cc:465-471)
 * or demodulatorResearch/ (gain used directly; WBFM default gain 64000/2pi) */
enum { SDR_SCALING_RADIODIAGS = 0, SDR_SCALING_RESEARCH = 1 };

/* sdr_accept_iq flags */
enum {
  SDR_IQ_HOST = 0,        /* iq points to host memory; the engine copies it to the GPU */
  SDR_IQ_DEVICE = 1,      /* iq points to device memory on the engine's GPU */
  SDR_IQ_U8_OFFSET = 0,   /* u8 offset-binary, not yet rotated: IqDataProcessor entry */
  SDR_IQ_S8_ROTATED = 2   /* signed, already Fs/4-rotated: demodulator entry, .iq file format */
};

enum {
  SDR_OK = 0,
  SDR_E_ARG = -1,      /* bad handle, channel, mode, kind, size or alignment */
  SDR_E_CUDA = -2,     /* CUDA runtime error (sdr_last_error has the text) */
  SDR_E_NOMEM = -3,
  SDR_E_TOO_LONG = -4, /* bytes_per_channel exceeds the engine's max_bytes_per_channel */
  SDR_E_FULL = -5,     /* ingest ring: every slot holds a tick that was not retired yet */
  SDR_E_EMPTY = -6     /* ingest ring: no tick in flight */
};

/* One engine = n_channels radios on CUDA device `device`. max_bytes_per_channel
 * bounds a single sdr_accept_iq (the reference block is 32768 bytes). All
 * channels start like a fresh reference object: mode None, gains 300 / 64000/2pi /
 * 256000/2pi / 300, LSB selected, all filter state zero. */
int sdr_engine_create(uint32_t n_channels, int device, uint64_t max_bytes_per_channel,
                      sdr_engine **out);
int sdr_engine_destroy(sdr_engine *e);

/* Run on a caller-owned cudaStream_t (NULL = the engine's own stream). */
int sdr_set_stream(sdr_engine *e, void *cuda_stream);
int sdr_set_scaling(sdr_engine *e, int scaling);

int sdr_set_mode(sdr_engine *e, uint32_t channel, int mode);
int sdr_set_modes(sdr_engine *e, const uint8_t *modes /* [n_channels] */);
int sdr_set_gain(sdr_engine *e, uint32_t channel, int kind, float gain);
int sdr_set_gain_all(sdr_engine *e, int kind, float gain);
int sdr_reset(sdr_engine *e, uint32_t channel, int kind);

/* Squelch (IqDataProcessor's Squelch object, Squelch.cc:227-273). A channel's block is
 * demodulated only if its mean magnitude, in dBFS minus the tuner gain, reaches the
 * threshold, or did so on the previous block (one-block tail); a squelched channel
 * produces no PCM (counts[ch] = 0) and its demodulator state does not advance. The
 * default threshold of -200 dBFS never closes (IqDataProcessor.cc:41). The decision is
 * per sdr_accept_iq call, as the reference's is per acceptIqData call. */
int sdr_set_squelch_threshold(sdr_engine *e, uint32_t channel, int32_t threshold_dbfs);
int sdr_set_receive_gain_db(sdr_engine *e, uint32_t channel, uint32_t gain_db);
/* Compute the signal state and mean magnitude of every call even while no threshold can
 * close (what enableSignalNotification / enableSignalMagnitudeNotification ask for). */
int sdr_enable_signal_reports(sdr_engine *e, int on);
/* Gate and mean magnitude of the last call, [n_channels] each; either may be NULL.
 * Synchronises. Fails with SDR_E_ARG if the last call did not run the squelch. */
int sdr_get_signal(sdr_engine *e, uint8_t *allowed, uint32_t *magnitude);

/* IQ dump (IqDataProcessor.cc:756-760): keep, for the channels it is enabled on, the block
 * of each sdr_accept_iq call as the reference hands it to UdpClient::sendData -- signed,
 * Fs/4-rotated interleaved I,Q, the .iq file / wire format (demod.cc:8-11) -- whatever the
 * squelch decides. The reference sends it as consecutive datagrams of at most 2048 bytes
 * (UdpClient.cc:77, 199-231); the caller slices. Enabling takes effect at the next call. */
int sdr_set_iq_dump(sdr_engine *e, uint32_t channel, int on);
/* The last call's dump of one channel: *n_bytes = bytes_per_channel of that call. out may be
 * NULL to ask for the size only. Synchronises. SDR_E_ARG if the channel was not dumped. */
int sdr_get_iq_dump(sdr_engine *e, uint32_t channel, int8_t *out, uint64_t capacity, uint64_t *n_bytes);
/* Device-resident dump of the last call: n_rows rows, row_stride apart, in ascending channel
 * order of the enabled channels. */
int sdr_iq_dump_device(sdr_engine *e, int8_t **rows, uint64_t *row_stride, uint32_t *n_rows);

/* One block for every channel: iq is [n_channels][channel_stride] bytes of
 * interleaved I,Q of which the first bytes_per_channel are consumed.
 * bytes_per_channel must be a multiple of 64 (one PCM sample); pointers and
 * stride multiples of 16. Asynchronous: returns once the work is queued; a caller
 * that queues faster than the GPU retires is held while 32 calls are in flight. Each
 * channel is demodulated by the mode it is in, exactly as the reference's
 * switch does; channels in mode None produce nothing. Filter state carries
 * over to the next call. */
int sdr_accept_iq(sdr_engine *e, const void *iq, uint64_t bytes_per_channel,
                  uint64_t channel_stride, uint32_t flags);

/* PCM of the last sdr_accept_iq: row ch holds counts[ch] samples (bytes/64, or 0
 * in mode None), rows are samples_per_row = bytes_per_channel/64 apart.
 * Synchronises. Either pointer may be NULL. */
int sdr_get_pcm(sdr_engine *e, int16_t *pcm, uint32_t *counts);
/* Device-resident PCM of the last call: [n_channels][*stride] int16. The engine alternates
 * between two buffers, so ask again after every sdr_accept_iq. */
int sdr_pcm_device(sdr_engine *e, int16_t **pcm, uint64_t *stride);
int sdr_sync(sdr_engine *e);
/* The engine runs part of its work on a second, internal stream. sdr_join makes the
 * engine's (or the caller's, see sdr_set_stream) stream wait for it without blocking the
 * host, so that an event recorded on that stream afterwards covers everything queued so
 * far. sdr_get_pcm and sdr_sync imply it. */
int sdr_join(sdr_engine *e);

/* Ingest ring: the bank's DataConsumer (DataConsumer.cc:220-352). A tick is one block of
 * every channel. The ring has n_slots pinned host slots of [n_channels][block_bytes]; a
 * committed tick's host->device copy, demodulation and PCM read-back are queued on three
 * streams and overlap those of its neighbours. Ticks retire in order. While a ring is in
 * use, feed the engine only through it. */
typedef struct sdr_ingest sdr_ingest;
int sdr_ingest_create(sdr_engine *e, uint32_t n_slots /* 2..64 */, uint64_t block_bytes, sdr_ingest **out);
int sdr_ingest_destroy(sdr_ingest *q);
/* DataConsumer::acceptData for the bank: copies iq ([n_channels][channel_stride], the first
 * bytes_per_channel of each row) into the next slot and queues it. Like the reference, a
 * block longer than block_bytes is clipped and a shorter one counts as a short block
 * (DataConsumer.cc:238-246). flags: SDR_IQ_U8_OFFSET or SDR_IQ_S8_ROTATED. SDR_E_FULL if
 * no slot is free. */
int sdr_ingest_accept(sdr_ingest *q, uint32_t timestamp, const void *iq, uint64_t bytes_per_channel,
                      uint64_t channel_stride, uint32_t flags);
/* The same without the copy: write the tick straight into the slot (*iq, rows
 * *channel_stride apart), then commit it. */
int sdr_ingest_acquire(sdr_ingest *q, void **iq, uint64_t *channel_stride);
int sdr_ingest_commit(sdr_ingest *q, uint32_t timestamp, uint64_t bytes_per_channel, uint32_t flags);
/* Waits for the oldest tick in flight and returns its timestamp, its PCM (pinned host memory,
 * [n_channels][*samples_per_row]) and counts[n_channels]; the pointers stay valid until the
 * next sdr_ingest_acquire / sdr_ingest_accept. SDR_E_EMPTY if nothing is in flight. */
int sdr_ingest_retire(sdr_ingest *q, uint32_t *timestamp, const int16_t **pcm, uint32_t *samples_per_row,
                      const uint32_t **counts);
/* lastTimeStamp and shortBlockCount (DataConsumer.cc:282-283), ticks committed, ticks in flight */
int sdr_ingest_stats(const sdr_ingest *q, uint32_t *last_timestamp, uint32_t *short_block_count, uint64_t *ticks,
                     uint32_t *in_flight);

/* ---- multi-device bank (SURVEY 8e) ----
 * n_channels radios over several GPUs of one box: device i of `devices` owns the contiguous
 * channels [n i / G, n (i + 1) / G) with an engine and an ingest ring of its own; nothing is
 * exchanged between devices. A tick is one block of every channel, written by the producer into
 * ONE pinned array [n_channels][block_bytes] (sdr_bank_acquire); sdr_bank_commit queues, per
 * device, the host->device copy of its slab, the demodulation and the copy of its PCM rows into
 * ONE pinned array [n_channels][bytes / 64] that sdr_bank_retire hands out once every device is
 * done. All calls only queue work, so one host thread drives the whole box. Calls on one bank
 * must be serialised by the caller. Setters not mirrored here go through the shard's engine
 * (sdr_bank_shard) with the channel index made local (channel - first_channel). */
typedef struct sdr_bank sdr_bank;
int sdr_bank_create(uint32_t n_channels, const int *devices, uint32_t n_devices, uint64_t block_bytes,
                    uint32_t n_slots /* 2..64 */, sdr_bank **out);
int sdr_bank_destroy(sdr_bank *b);
uint32_t sdr_bank_device_count(const sdr_bank *b);
/* Shard i: its CUDA device, first channel, channel count and engine; any pointer may be NULL. */
int sdr_bank_shard(const sdr_bank *b, uint32_t i, int *device, uint32_t *first_channel, uint32_t *n_channels,
                   sdr_engine **engine);
int sdr_bank_set_mode(sdr_bank *b, uint32_t channel, int mode);
int sdr_bank_set_modes(sdr_bank *b, const uint8_t *modes /* [n_channels] */);
int sdr_bank_set_gain(sdr_bank *b, uint32_t channel, int kind, float gain);
int sdr_bank_reset(sdr_bank *b, uint32_t channel, int kind);
int sdr_bank_set_squelch_threshold(sdr_bank *b, uint32_t channel, int32_t threshold_dbfs);
/* The next free tick array, [n_channels][*channel_stride] bytes of pinned host memory. */
int sdr_bank_acquire(sdr_bank *b, void **iq, uint64_t *channel_stride);
/* Queue the acquired tick on every device (flags: SDR_IQ_U8_OFFSET or SDR_IQ_S8_ROTATED). A tick
 * longer than block_bytes is clipped, a shorter one counts as a short block on every shard. */
int sdr_bank_commit(sdr_bank *b, uint32_t timestamp, uint64_t bytes_per_channel, uint32_t flags);
/* Waits for the oldest tick in flight on every device: its PCM [n_channels][*samples_per_row]
 * (pinned host memory, valid until the slot is acquired again) and counts[n_channels]. */
int sdr_bank_retire(sdr_bank *b, uint32_t *timestamp, const int16_t **pcm, uint32_t *samples_per_row,
                    const uint32_t **counts);
/* Text of the last error on this bank (or of the last failed create if b is NULL). */
const char *sdr_bank_last_error(const sdr_bank *b);

/* ---- batched multirate filter banks (SURVEY 8(f)-4) ----
 * The reference's generic filter classes that the IQ->PCM path does not instantiate itself.
 * One bank = n_rows independent objects of one class with the same taps; a row is one object's
 * sample stream. Results are those of feeding the reference object the same samples one by one
 * (bit-identical: float taps accumulate in tap order with single-rounded multiply and add, the
 * Q15 classes quantise taps with round(h*32768) and clamp after every tap), however the stream
 * is cut into calls. factor = 1 makes a decimator the plain FirFilter / FirFilter_int16. */
typedef struct sdr_filter_bank sdr_filter_bank;
enum {
  SDR_FILTER_DECIMATOR_F32 = 1,     /* Filters/Decimator.cc (factor 1: Filters/FirFilter.cc) */
  SDR_FILTER_INTERPOLATOR_F32 = 2,  /* Filters/Interpolator.cc; n_taps must be a multiple of factor */
  SDR_FILTER_DECIMATOR_I16 = 3,     /* Filters/Int16/Decimator_int16.cc (factor 1: FirFilter_int16.cc) */
  SDR_FILTER_INTERPOLATOR_I16 = 4,  /* Filters/Int16/Interpolator_int16.cc */
  SDR_FILTER_IIR_F32 = 5            /* Filters/IirFilter.cc; created by sdr_filter_bank_create_iir only */
};
/* taps: the prototype filter h[0..n_taps-1] exactly as the reference constructor takes it. */
int sdr_filter_bank_create(int device, int kind, uint32_t n_rows, const float *taps, uint32_t n_taps,
                           uint32_t factor, sdr_filter_bank **out);
/* n_rows IirFilter(nb, b, na, a) objects (Direct Form I, float in and out): per sample
 *   fir = 0; fir = fir + b[k]*x[n-k] (k = 0 .. nb-1);  r = 0; r = r + a[0]*y[n-na];
 *   r = r + a[k]*y[n-k] (k = 1 .. na-1);  y[n] = fir - r
 * in that order, every operation single-rounded (note a[0] meets the OLDEST output, as in the
 * reference's ring walk). 1 <= nb <= 64, 1 <= na <= 8, 1 <= n_rows <= 65535; a run takes fewer than
 * 2^31 samples per row and produces n_in outputs per row. NaN bit patterns may differ from x86's. */
int sdr_filter_bank_create_iir(int device, uint32_t n_rows, const float *b, uint32_t nb, const float *a, uint32_t na,
                               sdr_filter_bank **out);
int sdr_filter_bank_destroy(sdr_filter_bank *b);
int sdr_filter_bank_set_stream(sdr_filter_bank *b, void *cuda_stream);
int sdr_filter_bank_reset(sdr_filter_bank *b);
/* Outputs per row a run of n_in samples per row will produce now: n_in * L for an interpolator,
 * n_in for an IIR bank, (pending + n_in) / M for a decimator (pending = samples a previous run left in the
 * reference's decimationBuffer, Decimator.cc:291-303). */
uint64_t sdr_filter_bank_out_count(const sdr_filter_bank *b, uint64_t n_in);
/* in: [n_rows][in_stride] elements (float or int16_t by kind), n_in used per row; out:
 * [n_rows][out_stride]. flags: SDR_IQ_HOST (copied in and out, returns when out is filled) or
 * SDR_IQ_DEVICE (queued on the bank's stream). *n_out = outputs written per row. */
int sdr_filter_bank_run(sdr_filter_bank *b, const void *in, uint64_t in_stride, uint64_t n_in, void *out,
                        uint64_t out_stride, uint64_t *n_out, uint32_t flags);
int sdr_filter_bank_sync(sdr_filter_bank *b);
/* The Q15 taps the int16 classes compute in their constructors (Decimator_int16.cc:58-62);
 * returns n_taps. SDR_E_ARG for an IIR bank (there is no Q15 IirFilter). */
int sdr_filter_bank_taps_q15(const sdr_filter_bank *b, int16_t *q);
uint64_t sdr_filter_bank_launch_count(const sdr_filter_bank *b);
const char *sdr_filter_bank_last_error(const sdr_filter_bank *b);

/* Launch shape of one demodulator kind: channels per CTA (1..32) and threads
 * per CTA (multiple of 32). 0 = let the engine choose. For tuning and tests. */
int sdr_set_launch_shape(sdr_engine *e, int kind, uint32_t channels_per_cta, uint32_t threads);
/* Kernels launched by this engine so far. */
uint64_t sdr_launch_count(const sdr_engine *e);
/* Bytes of continuation state one channel keeps for `kind`. */
int sdr_state_bytes(int kind);
/* Text of the last error on this engine (or of the last failed create if e is NULL). */
const char *sdr_last_error(const sdr_engine *e);
const char *sdr_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SDR_B200_H */
