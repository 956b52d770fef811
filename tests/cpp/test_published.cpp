// tests/cpp/test_published.cpp -- CPU-only.  mlb::PublishedSignal (include/mlb200_host.hpp) in lockstep with
// the reference's SignalProcessor::PublishedSignal (source/app/MLSignalProcessor.{h,cpp}, compiled in place)
// on random sequences of writeQuick / writeQuickVert / read / readLatest / peekLatest.
//
// Every value read back (counts, buffers, available frames) is hashed per run.  Built with -DHAVE_REFERENCE
// (the reference sources on the include path) the two classes also run in lockstep, and `record` writes the
// reference's hashes to the digest file; built without, mlb::PublishedSignal's hashes must equal the recorded ones.
//   test_published <digest file> [record]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "mlb200_host.hpp"
#include "lockstep_digest.h"
#ifdef HAVE_REFERENCE
#include "MLSignalProcessor.h"
#endif

static int g_fail = 0, g_checks = 0;
#define REQUIRE(c) do { ++g_checks; if (!(c)) { ++g_fail; std::printf("REQUIRE failed: %s line %d\n", #c, __LINE__); } } while (0)
static unsigned rnd(unsigned& s) { s = s * 1664525u + 1013904223u; return s >> 8; }

#ifdef HAVE_REFERENCE
#define REF(...) __VA_ARGS__
#else
#define REF(...) (void)0
#endif

template <size_t CH>
static void run(Digests& d, unsigned seed, int octaves, int maxFrames, int maxVoices)
{
  unsigned s = seed;
  REF(ml::SignalProcessor::PublishedSignal ref(maxFrames, maxVoices, (int)CH, octaves));
  mlb::PublishedSignal mine(maxFrames, maxVoices, (int)CH, octaves);
  Hash hr, hm;
  float counter = 0.f;
  std::vector<float> a(4096), b(4096);
  for (int step = 0; step < 600; ++step)
  {
    const unsigned op = rnd(s) % 6;
    if (op <= 2)
    {
      float v[CH * 64];
      for (size_t j = 0; j < CH; ++j)
        for (int n = 0; n < 64; ++n) v[j * 64 + n] = counter++;
      const size_t frames = 1 + rnd(s) % (size_t)std::min(64, maxFrames);
      REF(ml::DSPVectorArray<CH> rv; for (size_t j = 0; j < CH; ++j) for (int n = 0; n < 64; ++n) rv.row(j)[n] = v[j * 64 + n];
          ref.template writeQuick<CH>(rv, frames, 0));
      mine.writeQuick(v, frames, 0);
    }
    else if (op == 3)
    {
      float frame[CH];
      for (size_t j = 0; j < CH; ++j) frame[j] = counter++;
      REF(ref.writeQuickVert(frame, CH, 0));
      mine.writeQuickVert(frame, CH, 0);
    }
    else
    {
      const size_t want = rnd(s) % 40;
      std::fill(a.begin(), a.end(), -1.f);
      std::fill(b.begin(), b.end(), -1.f);
      size_t ra = 0, rb = 0;
      if (op == 4)
        REF(ra = ref.read(a.data(), want)), rb = mine.read(b.data(), want);
      else if (rnd(s) & 1)
        REF(ra = ref.readLatest(a.data(), want)), rb = mine.readLatest(b.data(), want);
      else
        REF(ref.peekLatest(a.data(), want)), mine.peekLatest(b.data(), want);
      REF(REQUIRE(ra == rb); REQUIRE(std::memcmp(a.data(), b.data(), a.size() * sizeof(float)) == 0));
      hr.add((uint64_t)ra), hr.add(a.data(), a.size() * sizeof(float));
      hm.add((uint64_t)rb), hm.add(b.data(), b.size() * sizeof(float));
    }
    REF(REQUIRE(ref.getReadAvailable() == mine.getReadAvailable());
        REQUIRE(ref.getAvailableFrames() == mine.getAvailableFrames());
        hr.add((uint64_t)ref.getReadAvailable()), hr.add((uint64_t)ref.getAvailableFrames()));
    hm.add((uint64_t)mine.getReadAvailable()), hm.add((uint64_t)mine.getAvailableFrames());
  }
  char name[64];
  std::snprintf(name, sizeof name, "published<%zu>/seed%u", CH, seed);
  REQUIRE(d.check(name, hr, hm));
}

int main(int argc, char** argv)
{
  if (argc < 2) { std::printf("usage: test_published <digest file> [record]\n"); return 2; }
  Digests d(argv[1], argc > 2 && std::strcmp(argv[2], "record") == 0, HAVE_REFERENCE_SOURCES);
  for (unsigned seed = 1; seed <= 6; ++seed)
  {
    run<1>(d, seed, 0, 64, 1);
    run<2>(d, seed, 2, 32, 4);
    run<3>(d, seed, 4, 16, 2);
    run<4>(d, seed, 1, 64, 8);
  }
  if (!d.finish()) ++g_fail;
  std::printf("%s: %d assertions, %d failed (%s)\n", g_fail ? "FAILED" : "ALL PASSED", g_checks, g_fail,
              HAVE_REFERENCE_SOURCES ? "in lockstep with the reference" : "against the reference's recorded digests");
  return g_fail ? 1 : 0;
}
