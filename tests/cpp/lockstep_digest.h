// tests/cpp/lockstep_digest.h -- hashes of what a lockstep test reads back from the reference's classes, so that
// the test can run without them: a digest file holds one "<run> <hash>" line per run, written from the reference
// (`record`, built with -DHAVE_REFERENCE) and checked against our classes everywhere.
#pragma once
#include <cstdint>
#include <cstdio>
#include <map>
#include <string>

#ifdef HAVE_REFERENCE
#define HAVE_REFERENCE_SOURCES 1
#else
#define HAVE_REFERENCE_SOURCES 0
#endif

struct Hash  // FNV-1a, 64 bit
{
  uint64_t h = 1469598103934665603ull;
  void add(const void* p, size_t n)
  {
    const unsigned char* c = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < n; ++i) h = (h ^ c[i]) * 1099511628211ull;
  }
  void add(uint64_t v) { add(&v, sizeof v); }
};

class Digests
{
 public:
  Digests(const char* path, bool record, bool haveReference) : path_(path), record_(record), haveRef_(haveReference)
  {
    if (record_ && !haveRef_) { std::printf("record needs the reference (-DHAVE_REFERENCE)\n"); ok_ = false; }
    if (record_) return;
    FILE* f = std::fopen(path, "r");
    if (!f) { std::printf("cannot read %s\n", path); ok_ = false; return; }
    char name[128];
    unsigned long long h;
    while (std::fscanf(f, "%127s %llx", name, &h) == 2) want_[name] = h;
    std::fclose(f);
  }

  // ref: the reference's hash (meaningful only with the reference); mine: ours.  Both must be the recorded one.
  bool check(const std::string& name, const Hash& ref, const Hash& mine)
  {
    if (record_)
    {
      want_[name] = ref.h;
      return ref.h == mine.h;
    }
    auto it = want_.find(name);
    if (it == want_.end()) { std::printf("%s: no recorded digest in %s\n", name.c_str(), path_.c_str()); return false; }
    bool good = mine.h == it->second && (!haveRef_ || ref.h == it->second);
    if (!good) std::printf("%s: digest differs from the recorded reference\n", name.c_str());
    return good;
  }

  bool finish()
  {
    if (!record_ || !ok_) return ok_;
    FILE* f = std::fopen(path_.c_str(), "w");
    if (!f) return false;
    for (auto& kv : want_) std::fprintf(f, "%s %016llx\n", kv.first.c_str(), (unsigned long long)kv.second);
    std::fclose(f);
    return true;
  }

 private:
  std::string path_;
  bool record_, haveRef_, ok_ = true;
  std::map<std::string, uint64_t> want_;
};
