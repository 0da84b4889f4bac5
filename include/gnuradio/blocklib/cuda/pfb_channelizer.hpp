// gr::cuda::pfb_channelizer_ccf -- M-channel polyphase analysis bank (SURVEY.md 8c): complex stream in, one
// complex vector of `channels` per hop D = M / oversample input items out (oversample 1: critically sampled;
// 2 or 4: GNU Radio's oversample_rate, see b200_pfb_params in b200dsp.h).
#pragma once
#include <gnuradio/blocklib/cuda/cuda_block.hpp>

namespace gr {
namespace cuda {

class pfb_channelizer_ccf : public block, public stream_owner
{
public:
    typedef std::shared_ptr<pfb_channelizer_ccf> sptr;
    // algorithm: 0 auto, 1 SIMT DFT, 2 DFT across branches as a tensor-core GEMM (b200_pfb_set_algorithm)
    static sptr make(size_t numchans, const std::vector<float>& taps, size_t channel_begin = 0,
                     size_t channel_count = 0, int algorithm = 0, int oversample = 1)
    {
        auto ptr = std::make_shared<pfb_channelizer_ccf>(numchans, taps, channel_begin, channel_count, oversample);
        if (algorithm)
            check(b200_pfb_set_algorithm(ptr->d_pfb, algorithm), "cuda::pfb_channelizer");
        ptr->add_port(port<gr_complex>::make("input", port_direction_t::INPUT));
        ptr->add_port(port<gr_complex>::make("output", port_direction_t::OUTPUT, { ptr->d_count }));
        return ptr;
    }
    pfb_channelizer_ccf(size_t numchans, const std::vector<float>& taps, size_t channel_begin, size_t channel_count,
                        int oversample = 1)
        : block("pfb_channelizer_ccf"), d_m(numchans), d_count(channel_count ? channel_count : numchans - channel_begin)
    {
        if (taps.size() % numchans)
            throw std::invalid_argument("pfb_channelizer: taps must be a multiple of numchans");
        b200_pfb_params p{};
        p.taps = taps.data();
        p.n_channels = (int32_t)numchans;
        p.taps_per_channel = (int32_t)(taps.size() / numchans);
        p.channel_begin = (int32_t)channel_begin;
        p.channel_count = (int32_t)channel_count;
        p.oversample = (int32_t)oversample;
        check(b200_pfb_create(&p, &d_pfb), "cuda::pfb_channelizer");
        int32_t os = 1;
        check(b200_pfb_get_oversample(d_pfb, &os), "cuda::pfb_channelizer");
        d_hop = d_m / (size_t)os;
    }
    ~pfb_channelizer_ccf() override { b200_pfb_destroy(d_pfb); }

    work_return_code_t work(std::vector<block_work_input>& work_input,
                            std::vector<block_work_output>& work_output) override
    {
        int64_t n_in = std::min<int64_t>(work_input[0].n_items, (int64_t)work_output[0].n_items * (int64_t)d_hop);
        int64_t nc = 0, nv = 0;
        if (n_in >= (int64_t)d_hop) {
            work_guard g(work_input, work_output, d_stream);
            check(b200_pfb_run(d_pfb, work_input[0].buffer->read_ptr(), work_output[0].buffer->write_ptr(), n_in,
                               &nc, &nv, d_stream),
                  "cuda::pfb_channelizer");
        }
        work_input[0].n_consumed = (int)nc;
        work_output[0].n_produced = (int)nv;
        return work_return_code_t::WORK_OK;
    }
    bool done() override
    {
        synchronize();
        return block::done();
    }

private:
    size_t d_m, d_count, d_hop = 0;
    b200_pfb* d_pfb = nullptr;
};

} // namespace cuda
} // namespace gr
