// GPU QA of the oversampled channelizer at flowgraph level: vector_source -> cuda::pfb_channelizer_ccf(oversample
// 2 / 4) -> vector_sink on small device rings, so the stream crosses many work() calls, ring wraps and frame splits
// at odd frames (the handle carries the history and the frame phase between calls).  Expected values: the fp64
// statement below.  Built and run by tests/test_pfb_oversampled_gpu.py.
#include <gnuradio/blocklib/blocks/vector_sink.hpp>
#include <gnuradio/blocklib/blocks/vector_source.hpp>
#include <gnuradio/blocklib/cuda/pfb_channelizer.hpp>
#include <gnuradio/cudabuffer.hpp>
#include <gnuradio/flowgraph.hpp>
#include <gnuradio/schedulers/mt/scheduler_mt.hpp>

#include <cmath>
#include <random>

#include "qa_common.hpp"

using namespace gr;

// fp64 reference, hop D, zeros before the stream (b200dsp.h):
//   u_i[t] = sum_r h[i + rM] x[tD + D-1-i-rM],  z_c[t] = sum_i u_{(i + tD) mod M}[t] e^{+j 2 pi i c / M}
static std::vector<gr_complex> reference(const std::vector<gr_complex>& x, const std::vector<float>& h, int M, int D)
{
    const int P = (int)(h.size() / M);
    const int64_t n_t = (int64_t)x.size() / D;
    std::vector<std::complex<double>> tw(M), u(M);
    for (int k = 0; k < M; k++)
        tw[k] = std::polar(1.0, 2.0 * M_PI * k / M);
    std::vector<gr_complex> y((size_t)n_t * M);
    for (int64_t t = 0; t < n_t; t++) {
        for (int i = 0; i < M; i++) {
            std::complex<double> a = 0;
            for (int r = 0; r < P; r++) {
                const int64_t n = t * D + D - 1 - i - (int64_t)r * M;
                if (n >= 0)
                    a += (double)h[i + r * M] * std::complex<double>(x[n]);
            }
            u[i] = a;
        }
        const int sh = (int)(t * D % M);
        for (int c = 0; c < M; c++) {
            std::complex<double> z = 0;
            for (int i = 0; i < M; i++)
                z += u[(i + sh) % M] * tw[(int64_t)i * c % M];
            y[(size_t)t * M + c] = gr_complex((float)z.real(), (float)z.imag());
        }
    }
    return y;
}

static std::vector<gr_complex> noise(size_t n, unsigned seed)
{
    std::mt19937 g(seed);
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    std::vector<gr_complex> v(n);
    for (auto& x : v)
        x = gr_complex(u(g), u(g));
    return v;
}

// random asymmetric prototype: a tap order mistake cannot hide behind symmetric taps
static std::vector<float> rtaps(size_t n, unsigned seed)
{
    std::mt19937 g(seed);
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    std::vector<float> v(n);
    for (auto& x : v)
        x = u(g) / std::sqrt((float)n);
    return v;
}

// per frame: relative RMS error < 1e-5 and worst channel < 1e-4 of the frame's RMS (all M reference channels)
static bool frames_ok(const std::vector<gr_complex>& y, const std::vector<gr_complex>& ref, int M, int cb, int cc)
{
    const size_t n = ref.size() / M;
    if (y.size() != n * cc) {
        std::printf("  got %zu items, want %zu\n", y.size(), n * cc);
        return false;
    }
    for (size_t t = 0; t < n; t++) {
        double e2 = 0, r2 = 0, worst = 0;
        for (int c = 0; c < M; c++)
            r2 += std::norm(std::complex<double>(ref[t * M + c]));
        for (int c = 0; c < cc; c++) {
            const double e = std::abs(std::complex<double>(y[t * cc + c]) - std::complex<double>(ref[t * M + cb + c]));
            if (!std::isfinite(e))
                return false;
            e2 += e * e;
            worst = std::max(worst, e);
        }
        const double rms = std::sqrt(r2 / M);
        if ((cc > 1 && std::sqrt(e2 / cc) >= 1e-5 * rms) || worst >= 1e-4 * rms) {
            std::printf("  frame %zu of %zu: rms error %.3g, worst %.3g, frame rms %.3g\n", t, n, std::sqrt(e2 / cc),
                        worst, rms);
            return false;
        }
    }
    return true;
}

static void run_case(int M, int P, int os, int cb, int cc, size_t n_in, unsigned seed)
{
    auto in = noise(n_in, seed);
    auto taps = rtaps((size_t)M * P, seed + 1);
    const int D = M / os;
    const auto exp = reference(in, taps, M, D);
    auto src = blocks::vector_source_c::make(in);
    auto ch = cuda::pfb_channelizer_ccf::make(M, taps, cb, cc, 0, os);
    const int n_ch = cc ? cc : M - cb;
    auto snk = blocks::vector_sink_c::make(n_ch);
    auto fg = flowgraph::make();
    fg->connect(src, 0, ch, 0)->set_custom_buffer(DEVICE_BUFFER_ARGS_SIZED(H2D, 2u << 20));
    fg->connect(ch, 0, snk, 0)->set_custom_buffer(DEVICE_BUFFER_ARGS_SIZED(D2H, 2u << 20));
    fg->set_scheduler(schedulers::scheduler_mt::make());
    fg->validate();
    fg->run();
    EXPECT_TRUE(frames_ok(snk->data(), exp, M, cb, n_ch));
}

// config 4's 64 channels at oversample 2: 3000017 items (not a whole number of frames), 93750 frames out
QA_TEST(Oversampled, Pfb64Os2)
{
    run_case(64, 16, 2, 0, 0, 3000017, 31);
}

// M = 16 at oversample 4 (hop 4) with a channel slice, 16-frame filters
QA_TEST(Oversampled, Pfb16Os4Slice)
{
    run_case(16, 16, 4, 3, 9, 1000003, 41);
}

// the oversampled bank refuses the tensor-core DFT form and the 8-channel kernels: an error, not a fallback
QA_TEST(Oversampled, Rejections)
{
    bool threw = false;
    try {
        cuda::pfb_channelizer_ccf::make(64, std::vector<float>(64 * 8, 0.1f), 0, 0, 2, 2);
    } catch (const std::exception&) {
        threw = true;
    }
    EXPECT_TRUE(threw);
    threw = false;
    try {
        cuda::pfb_channelizer_ccf::make(8, std::vector<float>(8 * 8, 0.1f), 0, 0, 0, 2);
    } catch (const std::exception&) {
        threw = true;
    }
    EXPECT_TRUE(threw);
}

int main(int argc, char** argv) { return qa_main(argc, argv); }
