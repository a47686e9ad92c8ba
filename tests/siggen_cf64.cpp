// tests/siggen_cf64.cpp — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// The synthetic FM-stereo + RDS generator of oracle/siggen.cpp before its uint8 quantisation:
// sig_generate_cf64 writes the same n samples x = xi + j xq as interleaved doubles (full scale 1).
// Bands whose stations span more dynamic range than uint8 holds, and captures in the channelizer's
// signed formats, are built from x. The parameters, the pulse table, the noise generator and the
// RDS chips are oracle/siggen.cpp's own (included below); the sample loop restates sig_generate's
// operation by operation, and tests/test_siggen_cf64.py proves the restatement exact: x quantised
// by the generator's rule clamp(round(127.5 + 127.5 x), 0, 255) equals sig_generate's bytes.
// Built by tests/signals.py with oracle/Makefile's flags for libsiggen.so.
#include "../oracle/siggen.cpp"

extern "C" {

int sig_generate_cf64(const sig_params *p, const uint8_t *bits, size_t n_bits, double *iq, size_t n) {
  if (!p || !iq || p->fs_iq <= 0) {
    return -1;
  }
  constexpr int kSpan = 5;
  constexpr int kOver = 1024;
  constexpr double kBeta = 0.8;
  static std::vector<float> table;
  if (table.empty()) {
    std::vector<float> t(static_cast<size_t>(2 * kSpan * kOver + 2));
    for (size_t i = 0; i < t.size(); i++) {
      t[i] = static_cast<float>(rrc(static_cast<double>(i) / kOver - kSpan, kBeta));
    }
    table.swap(t);
  }
  std::vector<int8_t> chips;
  if (n_bits > 0 && p->rds_amp != 0.0) {
    int ones = 0;
    for (size_t i = 0; i < n_bits; i++) {
      ones += bits[i] & 1;
    }
    const size_t reps = (ones % 2) ? 2 : 1;
    int e = 0;
    chips.reserve(2 * n_bits * reps);
    for (size_t r = 0; r < reps; r++) {
      for (size_t i = 0; i < n_bits; i++) {
        e ^= (bits[i] & 1);
        chips.push_back(e ? 1 : -1);
        chips.push_back(e ? -1 : 1);
      }
    }
  }
  const long n_chips = static_cast<long>(chips.size());
  const double chip_rate = 2375.0;
  const double wp = 2.0 * M_PI * 19000.0;
  const double dt = 1.0 / p->fs_iq;
  const double sigma = (p->snr_db >= 200.0)
                           ? 0.0
                           : p->iq_amp * std::sqrt(0.5 / std::pow(10.0, p->snr_db / 10.0));
  Rng rng{p->seed * 0x2545f4914f6cdd1dULL + 0x1234567ULL};
  double phi = 0.0;
  const uint64_t first = p->start_sample;
  const uint64_t last = p->start_sample + n;
  for (uint64_t k = 0; k < last; k++) {
    const double t = static_cast<double>(k) * dt;
    const double l = p->tone_l_amp * std::sin(2.0 * M_PI * p->tone_l_hz * t);
    const double r = p->tone_r_amp * std::sin(2.0 * M_PI * p->tone_r_hz * t);
    double mm = p->audio_gain * (l + r) + p->audio_gain * (l - r) * std::sin(2.0 * wp * t) +
                p->pilot_amp * std::sin(wp * t);
    if (n_chips > 0) {
      const double u = t * chip_rate;
      const long c0 = static_cast<long>(std::floor(u));
      double d = 0.0;
      for (int j = -kSpan + 1; j <= kSpan; j++) {
        const long ci = c0 + j;
        const double z = u - static_cast<double>(ci);
        const double pos = (z + kSpan) * kOver;
        const long ip = static_cast<long>(pos);
        const double fr = pos - static_cast<double>(ip);
        const double pv = table[static_cast<size_t>(ip)] * (1.0 - fr) +
                          table[static_cast<size_t>(ip) + 1] * fr;
        long cm = ci % n_chips;
        if (cm < 0) {
          cm += n_chips;
        }
        d += chips[static_cast<size_t>(cm)] * pv;
      }
      mm += p->rds_amp * d * std::sin(3.0 * wp * t);
    }
    phi += 2.0 * M_PI * (p->deviation * mm + p->freq_offset_hz) * dt;
    if (phi > M_PI) {
      phi -= 2.0 * M_PI;
    } else if (phi < -M_PI) {
      phi += 2.0 * M_PI;
    }
    double n1 = 0.0, n2 = 0.0;
    if (sigma > 0.0) {
      rng.gauss2(&n1, &n2);
    }
    if (k < first) {
      continue;
    }
    const size_t o = static_cast<size_t>(k - first) * 2;
    iq[o] = p->iq_amp * std::cos(phi) + p->dc_i + sigma * n1;
    iq[o + 1] = p->iq_amp * std::sin(phi) + p->dc_q + sigma * n2;
  }
  return 0;
}

}  // extern "C"
