// tests/cpp/test_ringbuffer.cpp -- CPU-only.  mlb::DSPBuffer and mlb::BatchedSignalProcessBuffer
// (include/mlb200_host.hpp) must behave like the reference's ml::DSPBuffer / ml::SignalProcessBuffer.
// The ring is driven on random operation sequences, and the batched process buffer is compared with a
// restatement of the reference's per-vector loop (MLSignalProcessBuffer.cpp:57-78) built from the reference's
// DSPBuffer.  Everything read back is hashed per run (tests/cpp/lockstep_digest.h): built with -DHAVE_REFERENCE
// (the reference sources on the include path) the reference's classes also run in lockstep and `record` writes
// their hashes; built without, our hashes must equal the recorded ones.  Mirrors Tests/dspBufferTest.cpp.
//   test_ringbuffer <digest file> [record]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "mlb200_host.hpp"
#include "lockstep_digest.h"
#ifdef HAVE_REFERENCE
#include "MLDSPBuffer.h"
#define REF(...) __VA_ARGS__
#else
#define REF(...) (void)0
#endif

static int g_fail = 0, g_checks = 0;
#define REQUIRE(c) do { ++g_checks; if (!(c)) { ++g_fail; std::printf("REQUIRE failed: %s line %d\n", #c, __LINE__); } } while (0)

static unsigned rnd(unsigned& s) { s = s * 1664525u + 1013904223u; return s >> 8; }

int main(int argc, char** argv)
{
  if (argc < 2) { std::printf("usage: test_ringbuffer <digest file> [record]\n"); return 2; }
  Digests d(argv[1], argc > 2 && std::strcmp(argv[2], "record") == 0, HAVE_REFERENCE_SOURCES);
  // ---- basic semantics (Tests/dspBufferTest.cpp: sizes, wrap, overflow) ----
  {
    mlb::DSPBuffer b;
    REQUIRE(b.resize(100) == 128);
    REQUIRE(mlb::DSPBuffer(10).getWriteAvailable() == 64);  // never below one vector
    std::vector<float> x(300), y(300, -1.f);
    for (int i = 0; i < 300; ++i) x[i] = (float)i;
    b.write(x.data(), 100);
    REQUIRE(b.getReadAvailable() == 100);
    REQUIRE(b.read(y.data(), 60) == 60 && y[59] == 59.f);
    b.write(x.data() + 100, 80);  // wraps
    REQUIRE(b.getReadAvailable() == 120);
    b.write(x.data() + 180, 20);  // overflows by 12: the oldest samples go
    REQUIRE(b.getReadAvailable() == 128);
    REQUIRE(b.read(y.data(), 1000) == 128 && y[0] == 72.f && y[127] == 199.f);
    float v[64];
    REQUIRE(!b.readVector(v) && v[0] == 0.f);  // silence, nothing consumed
  }
  // ---- lockstep with the reference's DSPBuffer on random operation sequences ----
  for (unsigned seed = 1; seed <= 20; ++seed)
  {
    unsigned s = seed;
    REF(ml::DSPBuffer ref);
    mlb::DSPBuffer mine;
    Hash hr, hm;
    const int size = 64 + (int)(rnd(s) % 900);
    const size_t cap = mine.resize(size);
    REF(REQUIRE(ref.resize(size) == cap); hr.add((uint64_t)cap));
    hm.add((uint64_t)cap);
    std::vector<float> src(4096), a(4096), b(4096);
    float counter = 0;
    for (int step = 0; step < 400; ++step)
    {
      const unsigned op = rnd(s) % 5;
      const size_t n = rnd(s) % std::min<size_t>(300, mine.getWriteAvailable() + mine.getReadAvailable() + 1);  // <= capacity
      if (op <= 1)
      {
        for (size_t i = 0; i < n; ++i) src[i] = counter++;
        REF(ref.write(src.data(), n));
        mine.write(src.data(), n);
      }
      else if (op == 2)
      {
        const size_t rb = mine.read(b.data(), n);
        REF(const size_t ra = ref.read(a.data(), n); REQUIRE(ra == rb);
            for (size_t i = 0; i < ra; ++i) REQUIRE(a[i] == b[i]);
            hr.add((uint64_t)ra), hr.add(a.data(), ra * sizeof(float)));
        hm.add((uint64_t)rb), hm.add(b.data(), rb * sizeof(float));
      }
      else if (op == 3)
      {
        float mv[64];
        mine.readVector(mv);
        REF(ml::DSPVector rv = ref.read(); for (int i = 0; i < 64; ++i) REQUIRE(rv[i] == mv[i]);
            hr.add(rv.getConstBuffer(), 64 * sizeof(float)));
        hm.add(mv, sizeof mv);
      }
      else
      {
        REF(ref.discard(n));
        mine.discard(n);
      }
      REF(REQUIRE(ref.getReadAvailable() == mine.getReadAvailable()); hr.add((uint64_t)ref.getReadAvailable()));
      hm.add((uint64_t)mine.getReadAvailable());
    }
    REQUIRE(d.check("ring/seed" + std::to_string(seed), hr, hm));
  }
  // ---- overlap-add writer / overlapping reader in lockstep (MLDSPBuffer.h:288-340): windowed frames of
  // `win` samples hopped by win - overlap, as an STFT resynthesis would use them ----
  for (unsigned seed = 1; seed <= 12; ++seed)
  {
    unsigned s = seed * 7919u;
    REF(ml::DSPBuffer ref);
    mlb::DSPBuffer mine;
    Hash hr, hm;
    const int size = 256 + (int)(rnd(s) % 2000);
    const size_t cap = mine.resize(size);
    REF(REQUIRE(ref.resize(size) == cap); hr.add((uint64_t)cap));
    hm.add((uint64_t)cap);
    const size_t win = 16 + rnd(s) % 100, overlap = rnd(s) % win;
    std::vector<float> frame(win), a(4096), b(4096);
    float counter = 1.f;
    for (int step = 0; step < 300; ++step)
    {
      const unsigned op = rnd(s) % 3;
      if (op <= 1)
      {
        for (size_t i = 0; i < win; ++i) frame[i] = (counter += 0.5f);
        REF(ref.writeWithOverlapAdd(frame.data(), win, overlap));
        mine.writeWithOverlapAdd(frame.data(), win, overlap);
      }
      else
      {
        const size_t n = std::min<size_t>(win, mine.getReadAvailable() + overlap);
        if (n > overlap)
        {
          std::fill(a.begin(), a.begin() + win, -1.f);
          std::fill(b.begin(), b.begin() + win, -1.f);
          mine.readWithOverlap(b.data(), win, overlap);
          REF(ref.readWithOverlap(a.data(), win, overlap); for (size_t i = 0; i < win; ++i) REQUIRE(a[i] == b[i]);
              hr.add(a.data(), win * sizeof(float)));
          hm.add(b.data(), win * sizeof(float));
        }
      }
      REF(REQUIRE(ref.getReadAvailable() == mine.getReadAvailable());
          REQUIRE(ref.getWriteAvailable() == mine.getWriteAvailable());
          hr.add((uint64_t)ref.getReadAvailable()), hr.add((uint64_t)ref.getWriteAvailable()));
      hm.add((uint64_t)mine.getReadAvailable()), hm.add((uint64_t)mine.getWriteAvailable());
    }
    REQUIRE(d.check("overlap/seed" + std::to_string(seed), hr, hm));
  }
  // ---- batched process buffer vs the reference's per-vector loop ----
  {
    const int maxFrames = 1024;
    mlb::BatchedSignalProcessBuffer batched(1, 2, maxFrames);
    REF(ml::DSPBuffer rin, rout[2]; rin.resize(maxFrames); rout[0].resize(maxFrames), rout[1].resize(maxFrames));
    Hash hr, hm;
    float acc_ref = 0.f, acc_mine = 0.f;  // a stateful "processor": running sum + input
    unsigned s = 99;
    std::vector<float> xin(maxFrames), o0(maxFrames), o1(maxFrames), r0(maxFrames), r1(maxFrames);
    float t = 0.f;
    for (int call = 0; call < 200; ++call)
    {
      const int frames = 1 + (int)(rnd(s) % maxFrames);
      for (int i = 0; i < frames; ++i) xin[i] = (t += 0.25f);
      // reference loop (MLSignalProcessBuffer.cpp:47-86)
      REF(rin.write(xin.data(), frames);
          while ((int)rout[0].getReadAvailable() < frames)
          {
            ml::DSPVector in = rin.read(), a, b;
            for (int i = 0; i < 64; ++i) { acc_ref += 1.f; a[i] = acc_ref + in[i]; b[i] = -in[i]; }
            rout[0].write(a), rout[1].write(b);
          }
          rout[0].read(r0.data(), frames), rout[1].read(r1.data(), frames);
          hr.add(r0.data(), frames * sizeof(float)), hr.add(r1.data(), frames * sizeof(float)));
      // batched
      const float* ins[1] = {xin.data()};
      float* outs[2] = {o0.data(), o1.data()};
      batched.process(ins, outs, frames, [&](const float* in, float* out, int n) {
        for (int v = 0; v < n; ++v)
          for (int i = 0; i < 64; ++i)
          {
            acc_mine += 1.f;
            out[(v * 2 + 0) * 64 + i] = acc_mine + in[v * 64 + i];
            out[(v * 2 + 1) * 64 + i] = -in[v * 64 + i];
          }
      });
      REF(for (int i = 0; i < frames; ++i) { REQUIRE(o0[i] == r0[i]); REQUIRE(o1[i] == r1[i]); });
      hm.add(o0.data(), frames * sizeof(float)), hm.add(o1.data(), frames * sizeof(float));
    }
    REQUIRE(d.check("process_buffer", hr, hm));
    (void)acc_ref;
  }
  if (!d.finish()) ++g_fail;
  std::printf("(checked %s)\n", HAVE_REFERENCE_SOURCES ? "in lockstep with the reference's DSPBuffer"
                                                        : "against the reference's recorded digests");
  std::printf("%s: %d checks, %d failed\n", g_fail ? "FAILED" : "ALL PASSED", g_checks, g_fail);
  return g_fail ? 1 : 0;
}
