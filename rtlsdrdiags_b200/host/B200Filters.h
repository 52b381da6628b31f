// Drop-ins for the reference's generic filter classes (radioDiags/Filters/Decimator.h:28-42,
// Interpolator.h:35-49, FirFilter.h:21-27, IirFilter.h and the Int16/ twins) over the batched filter banks of
// the C ABI (sdr_filter_bank_*): same class names, constructors and per-sample methods, plus a
// BLOCK method each -- the per-sample methods run a one-sample bank call (correct, and as slow as
// that sounds); a caller that has a buffer should hand over the buffer, and a caller that has many
// streams should use a bank with one row per stream directly.
//
//   reference                                        here
//   Decimator(N, h, M) / Decimator_int16(N, h, M)    same; bool decimate(x, &y); uint32_t decimate(in, n, out)
//   Interpolator(N, h, L) / Interpolator_int16       same; void interpolate(x, yL); void interpolate(in, n, out)
//   FirFilter(N, h) / FirFilter_int16(N, h)          same; T filterData(x); void filterData(in, n, out)
//   IirFilter(nb, b, na, a)                          same; float filterData(x); void filterData(in, n, out)
//   resetFilterState()                               same
// Results are those of the reference classes fed the same samples one by one (bit-identical, see
// include/sdr_b200.h), however the stream is cut into calls.
#ifndef B200_FILTERS_H
#define B200_FILTERS_H

#include <stdint.h>

#include "../../include/sdr_b200.h"

template <class T, int KIND>
class B200FilterRow
{
  public:
  void resetFilterState(void) { sdr_filter_bank_reset(bank); }
  // status of the last bank call (SDR_OK or SDR_E_*); the reference's methods cannot fail
  int lastStatus(void) const { return status; }

  protected:
  B200FilterRow(int filterLength, float *coefficientsPtr, int factor)
  {
    bank = 0;
    status = sdr_filter_bank_create(0, KIND, 1, coefficientsPtr, (uint32_t)filterLength, (uint32_t)factor, &bank);
  } // B200FilterRow
  ~B200FilterRow(void)
  {
    if (bank != 0) sdr_filter_bank_destroy(bank);
  } // ~B200FilterRow
  // n input samples in, returns the number of output samples written
  uint32_t run(const T *in, uint32_t n, T *out, uint32_t outCapacity)
  {
    uint64_t produced = 0;
    if (bank == 0) return (0);
    status = sdr_filter_bank_run(bank, in, n, n, out, outCapacity, &produced, SDR_IQ_HOST);
    return (status == SDR_OK ? (uint32_t)produced : 0);
  } // run

  sdr_filter_bank *bank;
  int status;
};

template <class T, int KIND>
class B200Decimator : public B200FilterRow<T, KIND>
{
  public:
  B200Decimator(int filterLength, float *coefficientsPtr, int decimationFactor)
      : B200FilterRow<T, KIND>(filterLength, coefficientsPtr, decimationFactor), factor(decimationFactor) {}
  // Decimator.cc:281-322: true (and *outputSamplePtr set) on every decimationFactor-th call
  bool decimate(T inputSample, T *outputSamplePtr)
  {
    T y;
    if (this->run(&inputSample, 1, &y, 1) == 1)
    {
      *outputSamplePtr = y;
      return (true);
    } // if
    return (false);
  } // decimate
  // the same for a block: returns how many outputs were written (at most (pending + n) / factor)
  uint32_t decimate(const T *inputPtr, uint32_t n, T *outputPtr) { return (this->run(inputPtr, n, outputPtr, n / factor + 1)); }

  private:
  uint32_t factor;
};

template <class T, int KIND>
class B200Interpolator : public B200FilterRow<T, KIND>
{
  public:
  B200Interpolator(int filterLength, float *coefficientsPtr, int interpolationFactor)
      : B200FilterRow<T, KIND>(filterLength, coefficientsPtr, interpolationFactor), factor(interpolationFactor) {}
  // Interpolator.cc: interpolationFactor outputs per input sample
  void interpolate(T inputSample, T *outputBufferPtr) { this->run(&inputSample, 1, outputBufferPtr, factor); }
  void interpolate(const T *inputPtr, uint32_t n, T *outputPtr) { this->run(inputPtr, n, outputPtr, n * factor); }

  private:
  uint32_t factor;
};

template <class T, int KIND>
class B200Fir : public B200FilterRow<T, KIND>
{
  public:
  B200Fir(int filterLength, float *coefficientsPtr) : B200FilterRow<T, KIND>(filterLength, coefficientsPtr, 1) {}
  // FirFilter.cc:144-185 / FirFilter_int16.cc:151-213
  T filterData(T x)
  {
    T y = 0;
    this->run(&x, 1, &y, 1);
    return (y);
  } // filterData
  void filterData(const T *inputPtr, uint32_t n, T *outputPtr) { this->run(inputPtr, n, outputPtr, n); }
};

// IirFilter.cc: Direct Form I, nb numerator and na denominator taps (1 <= nb <= 64, 1 <= na <= 8)
class IirFilter
{
  public:
  IirFilter(int numberOfNumeratorTaps, float *numeratorTapsPtr, int numberOfDenominatorTaps, float *denominatorTapsPtr)
  {
    bank = 0;
    status = sdr_filter_bank_create_iir(0, 1, numeratorTapsPtr, (uint32_t)numberOfNumeratorTaps, denominatorTapsPtr,
                                        (uint32_t)numberOfDenominatorTaps, &bank);
  } // IirFilter
  ~IirFilter(void)
  {
    if (bank != 0) sdr_filter_bank_destroy(bank);
  } // ~IirFilter
  // zeroes the input and output histories
  void resetFilterState(void)
  {
    if (bank != 0) status = sdr_filter_bank_reset(bank);
  } // resetFilterState
  float filterData(float x)
  {
    float y = 0;
    filterData(&x, 1, &y);
    return (y);
  } // filterData
  void filterData(const float *inputPtr, uint32_t n, float *outputPtr)
  {
    uint64_t produced = 0;
    if (bank == 0) return;
    status = sdr_filter_bank_run(bank, inputPtr, n, n, outputPtr, n, &produced, SDR_IQ_HOST);
  } // filterData
  // status of the last bank call (SDR_OK or SDR_E_*); the reference's methods cannot fail
  int lastStatus(void) const { return status; }

  private:
  sdr_filter_bank *bank;
  int status;
};

typedef B200Decimator<float, SDR_FILTER_DECIMATOR_F32> Decimator;
typedef B200Decimator<int16_t, SDR_FILTER_DECIMATOR_I16> Decimator_int16;
typedef B200Interpolator<float, SDR_FILTER_INTERPOLATOR_F32> Interpolator;
typedef B200Interpolator<int16_t, SDR_FILTER_INTERPOLATOR_I16> Interpolator_int16;
typedef B200Fir<float, SDR_FILTER_DECIMATOR_F32> FirFilter;
typedef B200Fir<int16_t, SDR_FILTER_DECIMATOR_I16> FirFilter_int16;

#endif // B200_FILTERS_H
