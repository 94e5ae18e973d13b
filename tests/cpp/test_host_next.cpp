// CPU-only tests of the SURVEY section 8(f) host pieces: the config loader with its expression grammar
// (include/srtb/program_options.hpp), the NPY writer, and the file reader's block/overlap arithmetic.
#include <chrono>
#include <cmath>
#include <complex>
#include <cstdio>
#include <filesystem>
#include <fstream>
#include <string>
#include <thread>
#include <vector>

#include "srtb/io/npy.hpp"
#include "srtb/io/udp_block_assembler.hpp"
#include "srtb/program_options.hpp"

#define CHECK(...)                                                                     \
  do {                                                                                 \
    if (!(__VA_ARGS__)) {                                                              \
      std::fprintf(stderr, "CHECK failed: %s (%s:%d)\n", #__VA_ARGS__, __FILE__, __LINE__); \
      return 1;                                                                        \
    }                                                                                  \
  } while (0)

int main(int argc, char** argv) {
  using srtb::program_options::parse;
  // expressions that appear in the shipped cfg files (srtb_config.cfg:2-8, srtb_config_1644-4559.cfg:2-3,26-28)
  CHECK(parse("2 ** 30") == 1073741824.0);
  CHECK(parse("2 ** 11") == 2048.0);
  CHECK(parse("1405 + (64 / 2)") == 1437.0);
  CHECK(parse("1000 * 1e6") == 1e9);
  CHECK(parse("128 * 1e6") == 128e6);
  CHECK(parse("-478.80") == -478.80);
  CHECK(parse("-64") == -64.0);
  // grammar: precedence, right-associative **, unary signs, functions, constants, case-insensitive
  CHECK(parse("1 + 2 * 3") == 7.0);
  CHECK(parse("(1 + 2) * 3") == 9.0);
  CHECK(parse("2 ** 3 ** 2") == 512.0);
  CHECK(parse("-2 ** 2") == 4.0);  // unary minus is a primary: (-2) ** 2
  CHECK(parse("2 * -3") == -6.0);
  CHECK(parse("10 / 4") == 2.5);
  CHECK(std::abs(parse("pi") - M_PI) < 1e-15 && std::abs(parse("PI * 2") - 2 * M_PI) < 1e-15);
  CHECK(std::abs(parse("e") - M_E) < 1e-15);
  CHECK(parse("sqrt(16) + abs(-2)") == 6.0);
  CHECK(parse("max(2, 3) + min(2, 3) + pow(2, 10)") == 1029.0);
  CHECK(std::abs(parse("atan2(1, 1)") - M_PI / 4) < 1e-15);
  CHECK(parse("floor(2.7) + ceil(2.1) + log10(1000)") == 8.0);
  CHECK(parse(" 1.5e3 ") == 1500.0);
  for (const char* bad : {"", "2 **", "1 +", "(1", "foo", "2 2", "sqrt 4", "max(1)"}) {
    bool threw = false;
    try {
      parse(bad);
    } catch (const std::invalid_argument&) {
      threw = true;
    }
    CHECK(threw);
  }
  // config text with the same keys and expression styles as the J1644 cfg
  const std::string cfg_text =
      "# example\n"
      "baseband_input_count = 2 ** 30\n"
      "spectrum_channel_count = 2 ** 11\n"
      "baseband_output_file_prefix = /dev/shm/\n"
      "log_level = 4\n"
      "mitigate_rfi_average_method_threshold = 1.5\n"
      "mitigate_rfi_spectral_kurtosis_threshold = 1.05\n"
      "signal_detect_signal_noise_threshold = 8\n"
      "signal_detect_max_boxcar_length = 256\n"
      "gui_enable = 1\n"
      "input_file_path = /tmp/buf3.bin   # comment\n"
      "baseband_input_bits = 2\n"
      "dm = -478.80\n"
      "baseband_reserve_sample = 0\n"
      "baseband_freq_low = 1405 + (64 / 2)\n"
      "baseband_bandwidth = -64\n"
      "baseband_sample_rate = 128 * 1e6\n"
      "mitigate_rfi_freq_list = 1418-1422\n"
      "udp_receiver_port = 12004, 12005\n"
      "udp_receiver_address = 10.0.1.2,10.0.1.3\n";
  auto m = srtb::program_options::parse_config_text(cfg_text);
  srtb::configs c;
  srtb::program_options::apply_changed_configs(m, c);
  CHECK(c.baseband_input_count == (size_t{1} << 30) && c.spectrum_channel_count == 2048);
  CHECK(c.baseband_input_bits == 2 && c.baseband_freq_low == 1437.0f && c.baseband_bandwidth == -64.0f);
  CHECK(c.baseband_sample_rate == 128e6f && c.dm == -478.80f && c.baseband_reserve_sample == false);
  CHECK(c.mitigate_rfi_average_method_threshold == 1.5f && c.mitigate_rfi_spectral_kurtosis_threshold == 1.05f);
  CHECK(c.signal_detect_signal_noise_threshold == 8.0f && c.signal_detect_max_boxcar_length == 256);
  CHECK(c.mitigate_rfi_freq_list == "1418-1422" && c.input_file_path == "/tmp/buf3.bin");
  CHECK(c.baseband_output_file_prefix == "/dev/shm/" && c.gui_enable == true);
  CHECK(c.udp_receiver_port.size() == 2 && c.udp_receiver_port[1] == 12005);
  CHECK(c.udp_receiver_address.size() == 2 && c.udp_receiver_address[1] == "10.0.1.3");
  CHECK(srtb::log::current_level == srtb::log::levels::DEBUG);
  srtb::log::current_level = srtb::log::levels::WARNING;
  // the reference's two example configuration files, verbatim (argv[2] = the directory holding them, tests/golden):
  // srtb_config.cfg:2-22 and srtb_config_1644-4559.cfg:2-29 must load into srtb::configs unchanged
  if (argc > 2) {
    const std::string ref = argv[2];
    {
      std::string b0 = "prog", b1 = "--config_file_name", b2 = ref + "/srtb_config.cfg";
      char* bv[] = {b0.data(), b1.data(), b2.data()};
      srtb::configs r;
      srtb::program_options::apply_changed_configs(srtb::program_options::parse_arguments(3, bv, "none.cfg"), r);
      CHECK(r.baseband_input_count == (size_t{1} << 30) && r.spectrum_channel_count == 2048);
      CHECK(r.baseband_format_type == "simple" && r.baseband_input_bits == -8);
      CHECK(r.baseband_freq_low == 1000.0f && r.baseband_bandwidth == 500.0f && r.baseband_sample_rate == 1e9f);
      CHECK(r.baseband_reserve_sample == false && r.baseband_output_file_prefix == "/dev/shm/");
      CHECK(r.udp_receiver_address.size() == 1 && r.udp_receiver_address[0] == "10.0.1.2" && r.udp_receiver_port[0] == 12004);
      CHECK(r.udp_receiver_cpu_preferred.size() == 1 && r.udp_receiver_cpu_preferred[0] == 29 && r.dm == 0.0f);
      CHECK(r.mitigate_rfi_average_method_threshold == 5.0f && r.mitigate_rfi_spectral_kurtosis_threshold == 1.05f);
      CHECK(r.signal_detect_signal_noise_threshold == 8.0f && r.signal_detect_max_boxcar_length == 16);
    }
    {
      std::string b0 = "prog", b1 = "--config_file_name", b2 = ref + "/srtb_config_1644-4559.cfg";
      char* bv[] = {b0.data(), b1.data(), b2.data()};
      srtb::configs r;
      srtb::program_options::apply_changed_configs(srtb::program_options::parse_arguments(3, bv, "none.cfg"), r);
      CHECK(r.baseband_input_count == (size_t{1} << 30) && r.spectrum_channel_count == 2048 && r.baseband_input_bits == 2);
      CHECK(r.baseband_freq_low == 1437.0f && r.baseband_bandwidth == -64.0f && r.baseband_sample_rate == 128e6f);
      CHECK(r.dm == -478.80f && r.baseband_reserve_sample == false && r.mitigate_rfi_freq_list == "1418-1422");
      CHECK(r.mitigate_rfi_average_method_threshold == 1.5f && r.signal_detect_max_boxcar_length == 256);
      CHECK(r.input_file_path == "/tmp/buf3.bin" && r.input_file_offset_bytes == 0 && r.gui_enable == true);
    }
    srtb::log::current_level = srtb::log::levels::WARNING;
  }
  // command line beats the file; unknown keys are rejected
  const std::string dir = (argc > 1) ? argv[1] : "/tmp";
  const std::string cfg_path = dir + "/srtb_test.cfg";
  {
    std::ofstream f(cfg_path);
    f << "dm = 10\nspectrum_channel_count = 2 ** 15\n";
  }
  std::string a0 = "prog", a1 = "--config_file_name", a2 = cfg_path, a3 = "--dm=56.778", a4 = "--baseband_input_bits", a5 = "-8";
  char* av[] = {a0.data(), a1.data(), a2.data(), a3.data(), a4.data(), a5.data()};
  auto merged = srtb::program_options::parse_arguments(6, av, "does_not_exist.cfg");
  srtb::configs c2;
  srtb::program_options::apply_changed_configs(merged, c2);
  CHECK(c2.dm == 56.778f && c2.spectrum_channel_count == 32768 && c2.baseband_input_bits == -8);
  bool threw = false;
  try {
    srtb::program_options::parse_config_text("no_such_option = 1\n");
  } catch (const std::invalid_argument&) {
    threw = true;
  }
  CHECK(threw);
  // NPY writer: header layout numpy accepts (checked again from Python in tests/test_host_abi.py)
  std::vector<std::complex<float>> spec(6);
  for (int i = 0; i < 6; i++) spec[i] = {float(i), float(-i)};
  srtb::io::npy_save(dir + "/srtb_test.npy", spec.data(), {2, 3});
  std::vector<float> tim = {1.f, 2.f, 3.f};
  srtb::io::npy_save(dir + "/srtb_test_1d.npy", tim.data(), {3});
  std::ifstream f(dir + "/srtb_test.npy", std::ios::binary);
  std::string bytes((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  CHECK(bytes.size() % 8 == 0 && bytes.substr(1, 5) == "NUMPY" && (bytes.size() - 48) % 64 == 0);
  // ---- UDP-shaped stream: packet framing + counter-keyed block assembly with loss and reordering
  {
    using namespace srtb::io;
    using B = backend_registry::fastmb_roach2;
    constexpr size_t d = B::packet_payload_size - B::packet_header_size;
    CHECK(d == 4096);
    std::vector<std::byte> stream(d * 24);
    for (size_t i = 0; i < stream.size(); i++) stream[i] = static_cast<std::byte>((i * 2654435761u >> 13) & 0xff);
    auto packets = udp::frame_stream<B>(stream, /*first_counter=*/1000);
    CHECK(packets.size() == 24 && B::parse_counter(packets[5]) == 1005);
    udp::memory_packet_provider prov;
    for (size_t i = 0; i < packets.size(); i++) {
      if (i == 3 || i == 12 || i == 13) continue;             // lost packets
      if (i == 4) { prov.push(packets[5]); prov.push(packets[4]); continue; }  // 4 and 5 swapped (mid-block)
      if (i == 5) continue;
      prov.push(packets[i]);
    }
    udp::block_assembler<udp::memory_packet_provider, B> asmblr{std::move(prov)};
    std::vector<std::byte> block(d * 8);
    for (int blk = 0; blk < 3; blk++) {
      auto first = asmblr.receive(block);
      CHECK(first.has_value() && *first == 1000u + 8u * blk);
      for (size_t pkt = 0; pkt < 8; pkt++) {
        const size_t g = blk * 8 + pkt;
        const bool lost = (g == 3 || g == 12 || g == 13);
        for (size_t j = 0; j < d; j += 511) {
          const std::byte expect = lost ? std::byte{0} : stream[g * d + j];
          CHECK(block[pkt * d + j] == expect);
        }
      }
    }
    CHECK(asmblr.total_lost_packet_count == 3 && asmblr.total_received_packet_count == 21);
    CHECK(!asmblr.receive(block).has_value());                 // stream exhausted
    bool threw2 = false;
    std::vector<std::byte> odd(d * 2 + 1);
    try {
      asmblr.receive(odd);
    } catch (const std::invalid_argument&) {
      threw2 = true;
    }
    CHECK(threw2);
    // gznupsr_a1: 64-byte header, counter in VDIF words 6|7, 8192 data bytes
    using G = backend_registry::gznupsr_a1;
    std::vector<std::byte> gp(G::packet_payload_size);
    G::write_header(gp, 0x0123456789abcdefull);
    CHECK(G::parse_counter(gp) == 0x0123456789abcdefull && G::packet_payload_size - G::packet_header_size == 8192);
    CHECK(backend_registry::naocpsr_snap1::data_stream_count == 2);
  }
  {
    // synthetic live stream (BASELINE config #5): packets released at a target rate with a running counter; a consumer
    // that stalls for longer than the backlog loses packets, which the assembler zero-fills and counts
    using namespace srtb::io;
    using B = backend_registry::fastmb_roach2;
    constexpr size_t d = B::packet_payload_size - B::packet_header_size;
    std::vector<std::byte> payload(16 * d);
    for (size_t i = 0; i < payload.size(); i++) payload[i] = static_cast<std::byte>(1 + i % 251);
    const double rate = 40e6;  // bytes/s
    udp::paced_packet_provider<B> prov{payload, rate, 7000, /*backlog_bytes=*/64 * d};
    prov.run_for(0.5);
    udp::block_assembler<udp::paced_packet_provider<B>, B> a{std::move(prov)};
    std::vector<std::byte> block(32 * d);
    const auto t0 = std::chrono::steady_clock::now();
    size_t blocks = 0;
    uint64_t expect_first = 7000;
    bool stalled = false;
    while (auto first = a.receive(block)) {
      CHECK(*first == expect_first);   // blocks are counter-contiguous even across lost packets
      expect_first += 32;
      blocks++;
      if (blocks == 20 && !stalled) {  // stall for much longer than the 64-packet backlog lasts (6.5 ms at this rate)
        std::this_thread::sleep_for(std::chrono::milliseconds(60));
        stalled = true;
      }
    }
    const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    CHECK(dt > 0.45 && dt < 1.0);
    const double achieved = (double)(a.total_received_packet_count + a.total_lost_packet_count) * d / dt;
    CHECK(achieved > 0.8 * rate && achieved < 1.2 * rate);
    CHECK(a.total_lost_packet_count > 300 && a.total_lost_packet_count < 900);  // ~60 ms of a 9766 packet/s stream
    CHECK(a.provider.dropped_packets() >= a.total_lost_packet_count - 32);
  }
  std::printf("host next ok\n");
  return 0;
}
