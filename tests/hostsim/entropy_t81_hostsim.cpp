// Host build of the AC refinement of pyjpegdecoder_b200/csrc/bj_entropy.cuh under the T.81 correction rule
// (BJ_PHASE_T81_REFINE, compat="libjpeg-turbo").  TEST-ONLY: entropy_hostsim.cpp with one more entry point,
// hs_acrefine_stream_t81, which runs the same parse / apply orchestration as hs_acrefine_stream but applies the
// corrections by the T.81 rule (acrefine_block<true, true>, the instantiation acrefine_apply_kernel<true> runs).
// Never used by the product.
#include "entropy_hostsim.cpp"

extern "C" {

uint32_t hs_acrefine_stream_t81(const uint32_t* words, uint64_t n_words, uint64_t start_byte, uint64_t end_byte,
                                const SimScan* ss_, uint32_t nblk_stream, int16_t* coef) {
    ScanCtx c = make_ctx(*ss_);
    HostSrc src{words, n_words};
    const uint32_t* tab = ss_->lut + c.ac_tab[0];
    const uint32_t end_rel = (uint32_t)((end_byte - start_byte) * 8);
    std::vector<uint32_t> pos(nblk_stream);
    {   // the parse is the same under both rules: the non-zero masks do not depend on the correction rule
        std::vector<uint32_t> pre(BJ_ACR_WIN_BITS);
        uint32_t win_base = 0, pos_bits = 0, eob_run = 0;
        auto build = [&](uint32_t base) {
            win_base = base;
            for (uint32_t k = 0; k < BJ_ACR_WIN_BITS; k++) pre[k] = acrefine_predecode(src, start_byte * 8 + base + k, tab);
        };
        build(0);
        for (uint32_t cb = 0; cb < nblk_stream; cb += 32) {
            int nb = (int)std::min<uint32_t>(32, nblk_stream - cb);
            uint8_t tabs[32 * BJ_ACR_TAB_STRIDE];
            for (int i = 0; i < nb; i++)
                acrefine_build_table(nonzero_mask(coef + (size_t)(cb + i) * 64), c.ss, c.se, tabs + i * BJ_ACR_TAB_STRIDE);
            int i = 0;
            while (i < nb) {
                if (pos_bits > win_base + BJ_ACR_WIN_BITS - BJ_ACR_WIN_SLACK) build(pos_bits);
                uint32_t err = 0;
                i = acrefine_parse_window(pre.data(), win_base, win_base + BJ_ACR_WIN_BITS - BJ_ACR_WIN_SLACK, c, end_rel, tabs, i,
                                          nb, pos_bits, eob_run, pos.data() + cb, err);
                if (err) return err;
            }
        }
    }
    uint32_t err = 0;
    for (uint32_t b = nblk_stream; b-- > 0;) {
        BitReader<HostSrc> rd;
        rd.seek(&src, start_byte * 8, pos[b] & ~BJ_ACR_IN_EOBRUN);
        uint32_t eob_run = (pos[b] & BJ_ACR_IN_EOBRUN) ? 1u : 0u;
        int16_t* p = coef + (size_t)b * 64;
        err |= acrefine_block<true, true>(rd, c, tab, end_rel, nonzero_mask(p), eob_run, p);
    }
    return err;
}

}  // extern "C"
