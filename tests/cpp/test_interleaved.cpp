// C++ host layer, interleaved input: the golden long_message recording in both channels of one stereo s16 buffer,
// decoded as two streams by SameBatchReceiver::process_interleaved; both must print samedec's line for it.
// usage: test_interleaved <long_message.bin>     (raw s16le)
// Without a GPU it must fail loudly with SAME_ERR_NO_DEVICE (exit code 3).
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>

#include "same_receiver.hpp"

#define CHECK(c) do { if (!(c)) { std::fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)

int main(int argc, char** argv) {
  if (argc != 2) { std::fprintf(stderr, "usage: %s long.bin\n", argv[0]); return 2; }
  std::ifstream f(argv[1], std::ios::binary);
  std::vector<char> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  std::vector<int16_t> mono(raw.size() / 2);
  std::memcpy(mono.data(), raw.data(), mono.size() * 2);
  std::vector<int16_t> stereo(2 * mono.size());
  for (size_t n = 0; n < mono.size(); ++n) stereo[2 * n] = stereo[2 * n + 1] = mono[n];
  try {
    auto rx = same::SameReceiverBuilder::samedec(22050).build_batch(2);
    auto evs = rx.process_interleaved(stereo, 2);
    auto tail = rx.flush_samedec();
    for (uint32_t s = 0; s < 2; ++s) {
      std::vector<std::string> lines;
      for (auto* v : {&evs[s], &tail[s]}) for (auto& e : *v) if (auto m = e.message_ok()) lines.push_back(m->text);
      CHECK(lines.size() == 1);
      CHECK(lines[0].rfind("ZCZC-EAS-DMO-372088-091724-919623", 0) == 0 && lines[0].size() == 252);
      std::printf("stream %u: %s\n", s, lines[0].c_str());
    }
    // a bad map is refused with the channel named, and changes nothing
    try {
      rx.submit_interleaved(stereo.data(), SAME_FMT_S16, 2, mono.size(), {1, 1});
      CHECK(false);
    } catch (const same::EngineError& e) {
      CHECK(e.code == SAME_ERR_INVALID_ARG && std::strstr(e.what(), "channel 1") != nullptr);
    }
    std::printf("CPP_INTERLEAVED_OK\n");
    return 0;
  } catch (const same::EngineError& e) {
    std::fprintf(stderr, "%s\n", e.what());
    return e.code == SAME_ERR_NO_DEVICE ? 3 : 4;
  }
}
