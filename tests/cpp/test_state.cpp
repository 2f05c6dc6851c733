// C++ host-layer test of the portable stream state: a receiver cloned mid-recording (SameReceiver::clone, the
// reference's `SameReceiver: Clone`, receiver.rs:70) and the original both finish the recording and print the text
// samedec prints for it.
// usage: test_state <npt.bin> <expected header line>      (raw s16le file)
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iostream>

#include "same_receiver.hpp"

static std::vector<int16_t> read_s16(const char* path) {
  std::ifstream f(path, std::ios::binary);
  std::vector<char> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  std::vector<int16_t> out(raw.size() / 2);
  std::memcpy(out.data(), raw.data(), out.size() * 2);
  return out;
}
#define CHECK(c) do { if (!(c)) { std::fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)

static std::vector<std::string> texts(same::SameReceiver& r, const std::vector<int16_t>& rest) {
  std::vector<std::string> out;
  for (auto& m : r.iter_messages(rest)) out.push_back(m.text);
  while (auto m = r.flush()) out.push_back(m->text);
  return out;
}

int main(int argc, char** argv) {
  if (argc != 3) { std::fprintf(stderr, "usage: %s npt.bin expected\n", argv[0]); return 2; }
  try {
    const auto rec = read_s16(argv[1]);
    const std::string want = argv[2];
    auto a = same::SameReceiverBuilder::samedec(22050).build();
    // the first burst has been received (Searching, Reading, Burst, Assembling, NoCarrier); the header is not out yet
    const size_t cut = 30000;
    CHECK(a.iter_events(std::vector<int16_t>(rec.begin(), rec.begin() + cut)).size() == 5);
    auto b = a.clone();
    CHECK(b.input_sample_counter() == cut);
    CHECK(b.export_state() == a.export_state());
    const std::vector<int16_t> rest(rec.begin() + cut, rec.end());
    const auto ta = texts(a, rest), tb = texts(b, rest);
    CHECK(ta.size() == 1 && ta[0] == want);
    CHECK(tb == ta);
    CHECK(a.input_sample_counter() == b.input_sample_counter());
    std::printf("CPP_STATE_OK\n");
    return 0;
  } catch (const same::EngineError& e) {
    std::fprintf(stderr, "%s\n", e.what());
    return e.code == SAME_ERR_NO_DEVICE ? 3 : 4;
  }
}
