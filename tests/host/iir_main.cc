// Test driver for the IirFilter drop-in (rtlsdrdiags_b200/host/B200Filters.h):
//   iir_main <b taps file (float32)> <a taps file (float32)> <block|sample>   stdin -> stdout
// block: three uneven calls, then resetFilterState() and the whole input once more (both outputs
// are written); sample: filterData(x) one sample at a time.
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "B200Filters.h"

static std::vector<float> slurp(FILE *f)
{
  std::vector<float> v;
  float buf[1024];
  size_t n;
  while ((n = fread(buf, sizeof(float), 1024, f)) > 0) v.insert(v.end(), buf, buf + n);
  return v;
}

static bool load(const char *path, std::vector<float> &v)
{
  FILE *f = fopen(path, "rb");
  if (!f) return false;
  v = slurp(f);
  fclose(f);
  return true;
}

int main(int argc, char **argv)
{
  std::vector<float> b, a;
  if (argc < 4 || !load(argv[1], b) || !load(argv[2], a)) return 1;
  std::vector<float> x = slurp(stdin), y(x.size());
  const uint32_t n = (uint32_t)x.size();
  IirFilter f((int)b.size(), b.data(), (int)a.size(), a.data());
  if (f.lastStatus() != SDR_OK) return 2;
  if (!strcmp(argv[3], "block"))
  {
    const uint32_t c1 = n / 5, c2 = n / 2;
    f.filterData(x.data(), c1, y.data());
    f.filterData(x.data() + c1, c2 - c1, y.data() + c1);
    f.filterData(x.data() + c2, n - c2, y.data() + c2);
    fwrite(y.data(), sizeof(float), y.size(), stdout);
    f.resetFilterState();
    f.filterData(x.data(), n, y.data());
  }
  else
    for (uint32_t i = 0; i < n; i++) y[i] = f.filterData(x[i]);
  if (f.lastStatus() != SDR_OK) return 3;
  fwrite(y.data(), sizeof(float), y.size(), stdout);
  return 0;
}
