// b200_bank -- drives every GPU of one box from ONE host thread through the multi-device bank
// of the C ABI (include/sdr_b200.h, sdr_bank_*): the shape of Radio.cc's reader loop
// (Radio.cc:1871-1926) and DataConsumer::acceptData (DataConsumer.cc:220-262) for a bank of
// radios. No Python, no torch: this is what a C++ host links.
//
//   b200_bank [-n channels] [-g gpus] [-m am|fm|wbfm|ssb|mixed] [-b block_bytes] [-t ticks] [-s slots]
//             [-q squelch_dbfs] [-i k] [-k squelch_block_bytes]
//
// A tick is one block of every channel. The producer writes each tick in place into the bank's
// pinned tick array (here: synthetic offset-binary IQ, a noisy carrier per channel); the bank
// copies every device's slab to its GPU, demodulates it and copies the PCM rows back into one
// pinned PCM array. Prints the end-to-end rate and a checksum of all PCM.
//
// -q arms every radio's squelch at that threshold and turns the signal reports on: every retired
// tick then hands back its gate and mean magnitude per radio, what the reference's signal-state and
// signal-magnitude callbacks receive (IqDataProcessor.cc:771-790); the JSON line adds the open
// (radio, tick) pairs and the mean magnitude. -i k dumps the IQ of every k-th radio
// (IqDataProcessor.cc:756-760); the JSON line adds the dumped bytes. -k sets the squelch block on
// every shard (the reference's acceptIqData length, 32768 in Radio.cc): each tick is then gated
// block by block, and with -q the JSON line adds open_blocks, the open (radio, block) pairs.
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/sdr_b200.h"

static int die(const char *what, sdr_bank *b)
{
  fprintf(stderr, "%s: %s\n", what, sdr_bank_last_error(b));
  return 1;
} // die

int main(int argc, char **argv)
{
  uint32_t nChannels = 8192, nGpus = 1, ticks = 20, slots = 3, dumpEvery = 0;
  uint64_t blockBytes = 32768, squelchBlock = 0;
  const char *mode = "mixed";
  bool squelch = false;
  int32_t squelchDbfs = -200;

  for (int i = 1; i + 1 < argc; i += 2)
  {
    if (!strcmp(argv[i], "-n")) nChannels = (uint32_t)atol(argv[i + 1]);
    else if (!strcmp(argv[i], "-g")) nGpus = (uint32_t)atol(argv[i + 1]);
    else if (!strcmp(argv[i], "-m")) mode = argv[i + 1];
    else if (!strcmp(argv[i], "-b")) blockBytes = (uint64_t)atol(argv[i + 1]);
    else if (!strcmp(argv[i], "-t")) ticks = (uint32_t)atol(argv[i + 1]);
    else if (!strcmp(argv[i], "-s")) slots = (uint32_t)atol(argv[i + 1]);
    else if (!strcmp(argv[i], "-q")) { squelch = true; squelchDbfs = (int32_t)atol(argv[i + 1]); }
    else if (!strcmp(argv[i], "-i")) dumpEvery = (uint32_t)atol(argv[i + 1]);
    else if (!strcmp(argv[i], "-k")) squelchBlock = (uint64_t)atol(argv[i + 1]);
  } // for

  std::vector<int> devices(nGpus);
  for (uint32_t g = 0; g < nGpus; g++) devices[g] = (int)g;
  sdr_bank *bank = NULL;
  if (sdr_bank_create(nChannels, devices.data(), nGpus, blockBytes, slots, &bank)) return die("sdr_bank_create", NULL);

  // IqDataProcessor::setDemodulatorMode per radio (IqDataProcessor.cc:236-262)
  std::vector<uint8_t> modes(nChannels);
  for (uint32_t ch = 0; ch < nChannels; ch++)
  {
    if (!strcmp(mode, "am")) modes[ch] = SDR_MODE_AM;
    else if (!strcmp(mode, "fm")) modes[ch] = SDR_MODE_FM;
    else if (!strcmp(mode, "wbfm")) modes[ch] = SDR_MODE_WBFM;
    else if (!strcmp(mode, "ssb")) modes[ch] = (ch & 1) ? SDR_MODE_USB : SDR_MODE_LSB;
    else modes[ch] = (uint8_t)(1 + ch % 5);
  } // for
  if (sdr_bank_set_modes(bank, modes.data())) return die("sdr_bank_set_modes", bank);
  // IqDataProcessor::setSignalDetectThreshold and the signal notifications (IqDataProcessor.cc:284-295)
  if (squelch)
  {
    for (uint32_t ch = 0; ch < nChannels; ch++)
      if (sdr_bank_set_squelch_threshold(bank, ch, squelchDbfs)) return die("sdr_bank_set_squelch_threshold", bank);
    if (sdr_bank_enable_signal_reports(bank, 1)) return die("sdr_bank_enable_signal_reports", bank);
  } // if
  if (squelchBlock && sdr_bank_set_squelch_block_bytes(bank, squelchBlock))
    return die("sdr_bank_set_squelch_block_bytes", bank);
  // IqDataProcessor::enableIqDump on every k-th radio (IqDataProcessor.cc:633-669)
  if (dumpEvery)
    for (uint32_t ch = 0; ch < nChannels; ch += dumpEvery)
      if (sdr_bank_set_iq_dump(bank, ch, 1)) return die("sdr_bank_set_iq_dump", bank);

  // fill every slot once with a noisy carrier per channel (what the dongles would deliver)
  for (uint32_t s = 0; s < slots; s++)
  {
    void *iq;
    uint64_t stride;
    if (sdr_bank_acquire(bank, &iq, &stride)) return die("sdr_bank_acquire", bank);
    uint32_t lcg = 12345u + s;
    for (uint32_t ch = 0; ch < nChannels; ch++)
    {
      uint8_t *row = (uint8_t *)iq + (size_t)ch * stride;
      const double w = 2.0 * M_PI * (0.01 + 0.0001 * (ch % 97));
      for (uint64_t k = 0; k < blockBytes / 2; k++)
      {
        lcg = lcg * 1664525u + 1013904223u;
        row[2 * k] = (uint8_t)(128.0 + 60.0 * cos(w * (double)k) + (double)((lcg >> 24) & 3));
        row[2 * k + 1] = (uint8_t)(128.0 + 60.0 * sin(w * (double)k) + (double)((lcg >> 28) & 3));
      } // for
    } // for
    if (sdr_bank_commit(bank, s, blockBytes, SDR_IQ_U8_OFFSET)) return die("sdr_bank_commit", bank);
  } // for
  for (uint32_t s = 0; s < slots; s++)
    if (sdr_bank_retire(bank, NULL, NULL, NULL, NULL)) return die("sdr_bank_retire", bank);

  // the timed loop: commit a tick, retire the one two ticks back (radioApp.cc:103-111 is the sink)
  long long checksum = 0;
  unsigned long long openChannelTicks = 0, openBlocks = 0, dumpBytes = 0;
  double magnitudeSum = 0;
  const uint32_t inFlight = slots - 1;
  const std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  for (uint32_t k = 0; k < ticks + inFlight; k++)
  {
    if (k < ticks)
    {
      void *iq;
      if (sdr_bank_acquire(bank, &iq, NULL)) return die("sdr_bank_acquire", bank);
      if (sdr_bank_commit(bank, k, blockBytes, SDR_IQ_U8_OFFSET)) return die("sdr_bank_commit", bank);
    } // if
    if (k >= inFlight)
    {
      const int16_t *pcm;
      const uint32_t *counts;
      uint32_t ts, samples;
      if (sdr_bank_retire(bank, &ts, &pcm, &samples, &counts)) return die("sdr_bank_retire", bank);
      for (uint32_t ch = 0; ch < nChannels; ch += 61) checksum += pcm[(size_t)ch * samples + (ts % samples)] + counts[ch];
      // the per-tick callbacks: signal state and magnitude of every radio, then the IQ dump
      if (squelch)
      {
        const uint8_t *allowed;
        const uint32_t *magnitude;
        if (sdr_bank_retired_signal(bank, &allowed, &magnitude)) return die("sdr_bank_retired_signal", bank);
        for (uint32_t ch = 0; ch < nChannels; ch++)
        {
          openChannelTicks += allowed[ch];
          magnitudeSum += magnitude[ch];
        } // for
        // every block's signal state, in block order (the reference's callbacks once per block)
        uint32_t nBlocks;
        if (sdr_bank_retired_signal_blocks(bank, &allowed, &magnitude, &nBlocks))
          return die("sdr_bank_retired_signal_blocks", bank);
        for (size_t i = 0; i < (size_t)nBlocks * nChannels; i++) openBlocks += allowed[i];
      } // if
      if (dumpEvery)
      {
        const int8_t *rows;
        const uint32_t *channels;
        uint64_t rowStride, nBytes;
        uint32_t nRows;
        if (sdr_bank_retired_iq_dump(bank, &rows, &rowStride, &nBytes, &channels, &nRows))
          return die("sdr_bank_retired_iq_dump", bank);
        dumpBytes += (unsigned long long)nRows * nBytes;
        for (uint32_t r = 0; r < nRows; r += 61) checksum += rows[(size_t)r * rowStride + (ts % nBytes)] + channels[r];
      } // if
    } // if
  } // for
  const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  const double samples = (double)ticks * nChannels * (double)(blockBytes / 2);
  printf("{\"tool\": \"b200_bank\", \"gpus\": %u, \"channels\": %u, \"mode\": \"%s\", \"block_bytes\": %llu, \"ticks\": %u, "
         "\"seconds\": %.6f, \"e2e_msamples_per_s\": %.1f, \"host_to_device_gb_per_s\": %.2f, \"checksum\": %lld",
         nGpus, nChannels, mode, (unsigned long long)blockBytes, ticks, secs, samples / secs / 1e6,
         samples * 2.0 / secs / 1e9, checksum);
  if (squelch)
    printf(", \"squelch_dbfs\": %d, \"open_channel_ticks\": %llu, \"open_blocks\": %llu, \"mean_magnitude\": %.3f",
           (int)squelchDbfs, openChannelTicks, openBlocks, magnitudeSum / ((double)ticks * nChannels));
  if (squelchBlock) printf(", \"squelch_block_bytes\": %llu", (unsigned long long)squelchBlock);
  if (dumpEvery) printf(", \"dump_every\": %u, \"dump_bytes\": %llu", dumpEvery, dumpBytes);
  printf("}\n");
  sdr_bank_destroy(bank);
  return 0;
} // main
