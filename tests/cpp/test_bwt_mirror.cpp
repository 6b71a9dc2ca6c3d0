// C++ host-mirror test of sab200::bwt / sab200::inverse_bwt (sab200_suffix_array.hpp): the worked example, round
// trips on seeded texts, and the refusal of a transform of no text.  Needs a GPU at run time.
#include <cstdio>
#include <cstring>
#include <random>
#include <stdexcept>
#include <vector>

#include "sab200_suffix_array.hpp"

static int fails = 0;
#define EXPECT(c)                                                    \
    do {                                                             \
        if (!(c)) {                                                  \
            std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #c); \
            ++fails;                                                 \
        }                                                            \
    } while (0)

int main() {
    const auto* banana = reinterpret_cast<const std::uint8_t*>("banana");
    auto t = sab200::bwt(banana, 6);
    EXPECT(t.second == 4 && std::memcmp(t.first.data(), "annbaa", 6) == 0);
    EXPECT(sab200::inverse_bwt(t.first.data(), 6, 4) == std::vector<std::uint8_t>(banana, banana + 6));
    std::mt19937_64 rng(7);
    for (std::size_t n : {0u, 1u, 2u, 100u, 5000u, 300000u}) {
        for (unsigned sigma : {1u, 4u, 256u}) {
            std::vector<std::uint8_t> s(n);
            for (auto& c : s) c = (std::uint8_t)(rng() % sigma);
            auto u = sab200::bwt(s.data(), n);
            EXPECT(u.first.size() == n && (n == 0 ? u.second == 0 : u.second >= 1 && u.second <= n));
            EXPECT(sab200::inverse_bwt(u.first.data(), n, u.second) == s);
        }
    }
    bool refused = false;
    try {
        sab200::inverse_bwt(reinterpret_cast<const std::uint8_t*>("aa"), 2, 1);  // psi has a fixed point: no text
    } catch (const std::invalid_argument&) {
        refused = true;
    }
    EXPECT(refused);
    sab200_shutdown();
    std::printf(fails ? "bwt mirror: %d failure(s)\n" : "bwt mirror: all checks passed\n", fails);
    return fails ? 1 : 0;
}
