// tests/cpp/test_router.cpp -- mlb::VoiceRouter (include/mlb200_events.hpp) + the Voice bank against
// the COMPLETE reference EventsToSignals (oracle/_ref/libmle2s.so: the reference's own .cpp files).
// A MIDI phrase (notes with voice stealing, sustain pedal, pitch bend, CCs, note and channel pressure,
// all-notes-off; polyphonic and unison) goes (a) into ml::EventsToSignals and (b) through the router
// into per-voice event records and then through a Voice bank -- the C port on the CPU, or the CUDA bank
// when run with the argument "gpu".  All 8 rows of every voice must agree bit for bit.
//
// Built with -DHAVE_REFERENCE (linked with libmle2s.so) the reference runs beside ours and `record` writes the
// hash of its rows per phrase (tests/cpp/lockstep_digest.h); built without, our rows must have the recorded hash.
//   test_router <digest file> [gpu] [record]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "mlb200_events.hpp"
#include "lockstep_digest.h"

#ifdef HAVE_REFERENCE
#define REF(...) __VA_ARGS__
#else
#define REF(...) (void)0
#endif

extern "C" {
#ifdef HAVE_REFERENCE
struct mle2s_full;
mle2s_full* mle2s_full_create(float sr, int polyphony, float glideSeconds, float driftAmount, int unison, int mpe);
void mle2s_full_destroy(mle2s_full*);
void mle2s_full_add_event(mle2s_full*, int type, int channel, int sourceIdx, int time, float v1, float v2);
void mle2s_full_process(mle2s_full*, int start, float* out);
#endif
struct mlport_voice_bank;
mlport_voice_bank* mlport_bank_create(int V, float sr, const int32_t* voiceIndex, const float* glideSeconds,
                                      const float* driftAmount, const float* pitchBend, unsigned flags);
void mlport_bank_destroy(mlport_voice_bank*);
void mlport_bank_set_main_voices(mlport_voice_bank*, const int32_t* main_voice);
double mlport_bank_process(mlport_voice_bank*, int T, const mlb_voice_events* ev, float* out, int nthreads);
}

static uint32_t rng_state = 12345;
static uint32_t rnd() { return rng_state = rng_state * 1664525u + 1013904223u; }
static float rndf() { return (float)(rnd() >> 8) / 16777216.f; }

// an MPE phrase: every note on its own member channel (2..9); per-channel bend, pressure and CC 74; channel 1
// (the main channel) carries global bend and pressure
static std::vector<mlb::Event> make_mpe_phrase(int T, int seed)
{
  rng_state = 4242u + (uint32_t)seed * 7919u;
  std::vector<mlb::Event> ev;
  std::vector<int> held;  // channels in use
  auto push = [&](int type, int chan, int src, int time, float v1, float v2)
  {
    mlb::Event e;
    e.type = (uint8_t)type, e.channel = (uint8_t)chan, e.sourceIdx = (uint16_t)src, e.time = time, e.value1 = v1, e.value2 = v2;
    ev.push_back(e);
  };
  int next_chan = 2;
  for (int t = 0; t < T; ++t)
  {
    const int base = t * 64;
    if (rnd() % 3 == 0)
    {
      const int key = 40 + (int)(rnd() % 36), chan = next_chan;
      next_chan = next_chan == 9 ? 2 : next_chan + 1;
      push(mlb::kNoteOn, chan, key, base + (int)(rnd() % 64), key / 12.f, 0.2f + 0.8f * rndf());
      held.push_back(chan);
    }
    if (!held.empty() && rnd() % 4 == 0)
    {
      const size_t i = rnd() % held.size();
      push(mlb::kNoteOff, held[i], 60, base + (int)(rnd() % 64), 0.f, 0.f);
      held.erase(held.begin() + (long)i);
    }
    if (rnd() % 5 == 0) push(mlb::kPitchBend, 1 + (int)(rnd() % 9), 0, base + (int)(rnd() % 64), rndf() * 2.f - 1.f, 0.f);
    if (rnd() % 5 == 0) push(mlb::kChannelPressure, 1 + (int)(rnd() % 9), 0, base + (int)(rnd() % 64), rndf(), 0.f);
    if (rnd() % 6 == 0) push(mlb::kController, 2 + (int)(rnd() % 8), 74, base + (int)(rnd() % 64), rndf(), 0.f);
    if (rnd() % 9 == 0) push(mlb::kController, 2 + (int)(rnd() % 8), 16, base + (int)(rnd() % 64), rndf(), 0.f);
    if (rnd() % 11 == 0) push(mlb::kSustainPedal, 1, 0, base + (int)(rnd() % 64), (rnd() & 1) ? 1.f : 0.f, 0.f);
    if (rnd() % 13 == 0) push(mlb::kNotePressure, 2 + (int)(rnd() % 8), 60, base + (int)(rnd() % 64), rndf(), 0.f);  // ignored in MPE
  }
  return ev;
}

static std::vector<mlb::Event> make_phrase(int T, int seed)
{
  rng_state = 777u + (uint32_t)seed * 9176u;
  std::vector<mlb::Event> ev;
  std::vector<int> held;
  auto push = [&](int type, int src, int time, float v1, float v2)
  {
    mlb::Event e;
    e.type = (uint8_t)type, e.channel = 1, e.sourceIdx = (uint16_t)src, e.time = time, e.value1 = v1, e.value2 = v2;
    ev.push_back(e);
  };
  for (int t = 0; t < T; ++t)
  {
    const int base = t * 64;
    if (rnd() % 3 == 0)  // a note on (more keys than voices: stealing happens)
    {
      const int key = 40 + (int)(rnd() % 36);
      push(mlb::kNoteOn, key, base + (int)(rnd() % 64), key / 12.f, 0.2f + 0.8f * rndf());
      held.push_back(key);
    }
    if (!held.empty() && rnd() % 4 == 0)
    {
      const size_t i = rnd() % held.size();
      push(mlb::kNoteOff, held[i], base + (int)(rnd() % 64), 0.f, 0.f);
      held.erase(held.begin() + (long)i);
    }
    if (rnd() % 9 == 0) push(mlb::kSustainPedal, 0, base + (int)(rnd() % 64), (rnd() & 1) ? 1.f : 0.f, 0.f);
    if (rnd() % 5 == 0) push(mlb::kPitchBend, 0, base + (int)(rnd() % 64), rndf() * 2.f - 1.f, 0.f);
    if (rnd() % 6 == 0) push(mlb::kController, 16, base + (int)(rnd() % 64), rndf(), 0.f);
    if (rnd() % 7 == 0) push(mlb::kController, 73 + (int)(rnd() & 1), base + (int)(rnd() % 64), rndf(), 0.f);
    if (rnd() % 8 == 0 && !held.empty()) push(mlb::kNotePressure, held[rnd() % held.size()], base + (int)(rnd() % 64), rndf(), 0.f);
    if (rnd() % 10 == 0) push(mlb::kChannelPressure, 0, base + (int)(rnd() % 64), rndf(), 0.f);
    if (rnd() % 61 == 0)
    {
      push(mlb::kController, 123, base + (int)(rnd() % 64), 0.f, 0.f);  // all notes off
      held.clear();
    }
  }
  return ev;
}

static int run_case(Digests& d, int polyphony, bool unison, int seed, bool gpu, bool mpe = false)
{
  const int T = 400, P = polyphony;
  const float sr = 48000.f, glide = 0.03f, drift = 0.5f;
  const auto phrase = mpe ? make_mpe_phrase(T, seed) : make_phrase(T, seed);

  REF(mle2s_full* ref = mle2s_full_create(sr, P, glide, drift, unison ? 1 : 0, mpe ? 1 : 0));
  mlb::VoiceRouter router(P, mpe ? mlb::VoiceRouter::kMPE : mlb::VoiceRouter::kMIDI);
  const int NR = router.recordCount(), first = mpe ? 1 : 0;  // bank voices; index of the first channel voice
  router.setUnison(unison);
  for (const auto& e : phrase)
  {
    REF(mle2s_full_add_event(ref, e.type, e.channel, e.sourceIdx, e.time, e.value1, e.value2));
    router.addEvent(e);
  }
  std::vector<float> want((size_t)T * P * 8 * 64);
  std::vector<mlb_voice_events> recs((size_t)T * NR);
  int overflow = 0;
  for (int t = 0; t < T; ++t)
  {
    REF(mle2s_full_process(ref, t * 64, want.data() + (size_t)t * P * 8 * 64));  // [P][8][64]
    overflow += router.processVector(t * 64, recs.data() + (size_t)t * NR);
  }
  REF(mle2s_full_destroy(ref));
  if (overflow) { std::printf("  (phrase needs > %d note events per voice-vector %d times)\n", MLB_VOICE_MAX_EVENTS, overflow); return 1; }

  // bank voice b is reference voice b + (mpe ? 0 : 1); MPE: voice 0 = the main voice, MIDI bend range 7, the channel
  // voices use mpePitchBendRangeInSemitones_{24.f} (.cpp:422-428)
  std::vector<int32_t> idx(NR), mainv(NR, -1);
  std::vector<float> gs(NR, glide), da(NR, drift), pb(NR, mpe ? 24.f : 7.f);
  for (int i = 0; i < NR; ++i) idx[i] = i + (mpe ? 0 : 1);
  if (mpe)
  {
    pb[0] = 7.f;
    for (int i = 1; i < NR; ++i) mainv[i] = 0;
  }
  const unsigned bank_flags = mpe ? 0u : MLB_VOICES_MIDI;
  std::vector<float> got((size_t)T * 8 * NR * 64);  // [T][8][NR][64]
  if (gpu)
  {
    mlb_voices* vb = nullptr;
    if (mlb_voices_create(NR, sr, idx.data(), gs.data(), da.data(), pb.data(), bank_flags, &vb) != MLB_OK ||
        (mpe && mlb_voices_set_main_voices(vb, mainv.data()) != MLB_OK) ||
        mlb_voices_process_host(vb, recs.data(), got.data(), T, 0xFF) != MLB_OK)
    {
      std::printf("  GPU bank failed: %s\n", mlb_last_error());
      return 2;
    }
    mlb_voices_destroy(vb);
  }
  else
  {
    mlport_voice_bank* b = mlport_bank_create(NR, sr, idx.data(), gs.data(), da.data(), pb.data(), bank_flags);
    if (mpe) mlport_bank_set_main_voices(b, mainv.data());
    mlport_bank_process(b, T, recs.data(), got.data(), 1);
    mlport_bank_destroy(b);
  }
  size_t bad = 0, total = 0;  // word comparisons, with the reference beside ours
  double energy = 0;
  std::vector<float> ours(want.size());  // [T][P][8][64], the reference's layout
  for (int t = 0; t < T; ++t)
    for (int v = 0; v < P; ++v)
      for (int r = 0; r < 8; ++r)
        for (int n = 0; n < 64; ++n)
        {
          const float b = got[(((size_t)t * 8 + r) * NR + v + first) * 64 + n];
          ours[(((size_t)t * P + v) * 8 + r) * 64 + n] = b;
          REF(const float a = want[(((size_t)t * P + v) * 8 + r) * 64 + n];
              uint32_t ua, ub;
              std::memcpy(&ua, &a, 4), std::memcpy(&ub, &b, 4);
              if (ua != ub)
              {
                if (bad < 5) std::printf("  mismatch t=%d voice=%d row=%d n=%d: reference %g (%08x) ours %g (%08x)\n", t, v, r, n, a, ua, b, ub);
                ++bad;
              });
          ++total;
          if (r == 1) energy += b;
        }
  Hash hr, hm;
  REF(hr.add(want.data(), want.size() * sizeof(float)));
  hm.add(ours.data(), ours.size() * sizeof(float));
  const std::string name = std::string(mpe ? "mpe" : "midi") + "/P" + std::to_string(P) + (unison ? "/unison" : "/poly") +
                           "/seed" + std::to_string(seed);
  const bool recorded = d.check(name, hr, hm);
  std::printf("  %s polyphony %d %s seed %d: ", mpe ? "MPE " : "MIDI", P, unison ? "unison" : "poly", seed);
  REF(std::printf("%zu of %zu words differ from the reference, ", bad, total));
  std::printf("digest %s the reference's (gate sum %.1f, %zu events)\n", recorded ? "equals" : "DIFFERS FROM", energy,
              phrase.size());
  return (bad || !recorded) ? 1 : (energy > 10 ? 0 : 1);
}

int main(int argc, char** argv)
{
  if (argc < 2) { std::printf("usage: test_router <digest file> [gpu] [record]\n"); return 2; }
  bool gpu = false, record = false;
  for (int i = 2; i < argc; ++i) gpu |= std::strcmp(argv[i], "gpu") == 0, record |= std::strcmp(argv[i], "record") == 0;
  Digests d(argv[1], record, HAVE_REFERENCE_SOURCES);
  if (gpu && mlb_init(0) != MLB_OK)
  {
    std::printf("no device: %s\n", mlb_last_error());
    return 77;
  }
  int fails = 0;
  fails += run_case(d, 4, false, 1, gpu);
  fails += run_case(d, 8, false, 2, gpu);
  fails += run_case(d, 2, false, 3, gpu);
  fails += run_case(d, 4, true, 4, gpu);
  fails += run_case(d, 16, false, 5, gpu);
  fails += run_case(d, 8, false, 6, gpu, true);
  fails += run_case(d, 4, false, 7, gpu, true);
  fails += run_case(d, 15, false, 8, gpu, true);
  // ---- limits are reported, not hidden ----
  {
    mlb::VoiceRouter router(1);  // one voice: every note steals it
    for (int i = 0; i < 7; ++i)
    {
      mlb::Event e;
      e.type = mlb::kNoteOn, e.channel = 1, e.sourceIdx = (uint16_t)(50 + i), e.time = 5 * i, e.value1 = 4.f, e.value2 = 0.5f;
      router.addEvent(e);
    }
    mlb::Event off;
    off.type = mlb::kController, off.sourceIdx = 120, off.time = 40, off.value1 = 0.f;  // all sound off: not routed
    router.addEvent(off);
    mlb_voice_events rec[1];
    const int overflow = router.processVector(0, rec);
    const bool ok = overflow == 7 - MLB_VOICE_MAX_EVENTS && rec[0].n_events == MLB_VOICE_MAX_EVENTS &&
                    router.unsupportedEvents() == 1 && rec[0].type[0] == mlb::kNoteOn && rec[0].type[1] == mlb::kNoteRetrig;
    std::printf("  overflow and unsupported-event reporting: %s\n", ok ? "ok" : "WRONG");
    fails += ok ? 0 : 1;
  }
  if (!d.finish()) ++fails;
  std::printf(fails ? "FAILED\n" : "ALL PASSED\n");
  return fails ? 1 : 0;
}
