// bj_entropy.cuh -- per-thread logic of the entropy stage (Huffman / run-length / progressive
// bookkeeping), written as __host__ __device__ templates over a bit source so that the CPU test-suite
// (tests/hostsim) can drive exactly the code the CUDA kernels in bj_entropy.cu run.
//
// Reference being replaced (tbpaolini/PyJpegDecoder, jpeg_decoder.py):
//   bits_generator / get_bits   :654-695    bit reader (un-stuffing is done by bj_unstuff.cu)
//   next_huffval                :712-722    canonical Huffman decode, <= 16 bits
//   bin_twos_complement         :1636-1646  EXTEND
//   baseline_dct_scan           :805-866    DC difference + AC run/size loop (EOB 0x00, ZRL 0xF0)
//   progressive_dct_scan        :983-1057   DC first / DC refine
//                               :1120-1256  AC first with EOB runs
//                               :1100-1115, :1183-1198, :1209-1232, :1258-1292  AC refinement
//
// Parallel decomposition (new design, nothing like it exists in the reference): a stream (restart
// interval, or a whole scan) is cut into subsequences of BJ_SUBSEQ_BITS bits.  The decoder state at
// a subsequence boundary is (bit position, zig-zag index, slot in the MCU).  Huffman codes
// self-synchronise: a decoder started at a wrong state falls into step with the true one after a few
// symbols, so a speculative pass that starts one subsequence early yields, for almost every
// subsequence, its true entry state; a fix-up pass re-decodes the few that disagree with their
// predecessor's exit state until nothing changes (then all states are true by induction from the
// known state at the stream start).  Prefix sums of "blocks started per subsequence" and of the DC
// differences then give every subsequence its first block index and DC predictors, and a final
// pass writes whole 128-byte blocks.
#pragma once
#include <stdint.h>

#include "../../include/b200jpeg.h"
#include "bj_pixel_math.cuh"  // BJ_HD

namespace bj {

// ---- packed decoder state ------------------------------------------------------------------------
// bits 0..43 bit position in the un-stuffed buffer, 44..50 zig-zag index, 51..54 slot.
BJ_HD uint64_t pack_state(uint64_t pos, int z, int slot) {
    return pos | ((uint64_t)(uint32_t)z << 44) | ((uint64_t)(uint32_t)slot << 51);
}
BJ_HD uint64_t state_pos(uint64_t s) { return s & ((1ull << 44) - 1); }
BJ_HD int state_z(uint64_t s) { return (int)((s >> 44) & 127); }
BJ_HD int state_slot(uint64_t s) { return (int)((s >> 51) & 15); }

// ---- Huffman LUT entry (built by pyjpegdecoder_b200/huffman.py) ----------------------------------
// Fields are byte aligned so that each one is a single LOP/PRMT on the device:
//   direct:   byte 0 = L + (symbol & 15) (bits consumed by code + value; bit 7 clear)
//             byte 1 = zig-zag advance for baseline AC (run + 1; 64 for EOB; 16 for ZRL; 1 for DC)
//             byte 2 = code length L (0 = no such code; such entries have byte 0 = byte 1 = 1 so that a
//                      speculating decoder still makes progress)
//             byte 3 = symbol
//   indirect: bit 7 set, bits 8..23 = offset of a 128-entry second-level table (relative to the table)
// first level: 512 entries indexed by the next 9 bits; second level by the following 7 bits.
#if defined(__CUDA_ARCH__)
#define BJ_UNLIKELY(x) __builtin_expect(!!(x), 0)
#else
#define BJ_UNLIKELY(x) (x)
#endif
// byte k of a 32-bit word: one PRMT on the device
BJ_HD uint32_t byte_of(uint32_t e, int k) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(e, 0u, 0x4440u + (uint32_t)k);
#else
    return (e >> (8 * k)) & 0xFFu;
#endif
}
BJ_HD uint32_t lut_lookup(const uint32_t* tab, uint32_t peek16) {
    uint32_t e = tab[peek16 >> 7];
    // codes longer than 9 bits are rare symbols: a real branch, not seven predicated instructions per symbol
    if (BJ_UNLIKELY(e & 0x80u)) e = tab[((e >> 8) & 0xFFFFu) + (peek16 & 127u)];
    return e;
}
BJ_HD int ent_total(uint32_t e) { return (int)byte_of(e, 0); }
BJ_HD int ent_adv(uint32_t e) { return (int)byte_of(e, 1); }
BJ_HD int ent_len(uint32_t e) { return (int)byte_of(e, 2); }
BJ_HD int ent_sym(uint32_t e) { return (int)(e >> 24); }

// EXTEND (bin_twos_complement, :1636-1646)
BJ_HD int extend(uint32_t v, int n) { return (n == 0) ? 0 : ((v >> (n - 1)) ? (int)v : (int)v - ((1 << n) - 1)); }

// EXTEND of the n (1..16) bits that follow the first `skipn` bits of the look-ahead pk, branch-free: JPEG stores a
// negative value as the one's complement of its magnitude, so with m = all-ones when the leading bit is clear the
// value is ((bits ^ m) >> (32 - n)) with its sign flipped by m.  n == 0 must be handled by the caller.
BJ_HD int take_extend(uint32_t pk, int skipn, int n) {
    const uint32_t t = pk << skipn;
    const uint32_t m = ~(uint32_t)((int32_t)t >> 31);
    const uint32_t w = (t ^ m) >> (32 - n);
    return (int)((w ^ m) - m);
}

// ---- bit reader over big-endian 32-bit words -----------------------------------------------------
// Two 32-bit words (w0 = current, w1 = next) and the number of bits of w0 already consumed: the next
// 32 bits are one funnel shift away, consuming bits is an add, and a refill is one word fetch about
// every third symbol.  One symbol never needs more than 16 code bits + 15 value bits = 31 bits.
BJ_HD uint32_t funnel_left(uint32_t hi, uint32_t lo, int sh) {  // upper 32 bits of (hi:lo) << sh, 0 <= sh < 32
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, sh);
#else
    return sh ? (hi << sh) | (lo >> (32 - sh)) : hi;
#endif
}

template <class Src>
struct BitReader {
    const Src* src;
    uint32_t w0, w1;  // current and next word
    uint32_t w2;      // the word after: fetched one refill before it is needed, so its latency is off the symbol chain
    int o;            // bits of w0 consumed (0..31)
    uint32_t next;    // next word to fetch
    uint32_t rel;     // bit position relative to `base` (a stream is far below 2^32 bits)
    uint64_t base;    // absolute bit position of the stream start

    BJ_HDM void seek(const Src* s, uint64_t base_bit, uint32_t rel_bit) {
        src = s;
        base = base_bit;
        rel = rel_bit;
        const uint64_t p = base_bit + rel_bit;
        uint32_t w = (uint32_t)(p >> 5);
        o = (int)(p & 31);
        src->start(w);
        w0 = src->word(w);
        w1 = src->word(w + 1);
        w2 = src->word(w + 2);
        next = w + 3;
    }
    BJ_HDM uint64_t abs_pos() const { return base + rel; }
    BJ_HDM uint32_t peek32() const { return funnel_left(w0, w1, o); }
    BJ_HDM uint32_t peek16() const { return peek32() >> 16; }
    // n bits (1..16) that follow the first `skipn` bits (skipn + n <= 32)
    BJ_HDM uint32_t bits_after(int skipn, int n) const { return (peek32() << skipn) >> (32 - n); }
    BJ_HDM void skip_long(uint32_t n) {  // any n
        o += (int)n;
        rel += n;
        while (o >= 32) {
            o -= 32;
            w0 = w1;
            w1 = w2;
            w2 = src->word(next++);
        }
    }
    BJ_HDM void skip(int n) {  // n <= 32
        o += n;
        rel += (uint32_t)n;
        if (o >= 32) {
            o -= 32;
            w0 = w1;
            w1 = w2;
            w2 = src->word(next++);
        }
    }
};

// value bits of a symbol taken from an already fetched 32-bit look-ahead
BJ_HD uint32_t take_bits(uint32_t pk, int skipn, int n) { return (pk << skipn) >> (32 - n); }

// ---- per-scan context (shared memory on the device) ----------------------------------------------
struct ScanCtx {
    uint16_t dc_tab[BJ_MAX_SLOTS];    // table offsets inside the blob
    uint16_t ac_tab[BJ_MAX_SLOTS];
    uint8_t slot_comp[BJ_MAX_SLOTS];  // slot -> DC predictor index
    uint32_t tabs[BJ_MAX_SLOTS];      // dc_tab | ac_tab << 16 (one load per block instead of two); see ctx_finish()
    int nslots;
    int ss, se, al;
};
BJ_HD void ctx_finish(ScanCtx& c) {
    for (int i = 0; i < BJ_MAX_SLOTS; i++) c.tabs[i] = (uint32_t)c.dc_tab[i] | ((uint32_t)c.ac_tab[i] << 16);
}

struct SubCount {
    uint32_t blocks;  // blocks started (baseline / DC) or block advance (AC first) in the subsequence
    int32_t dc[3];    // sum of DC differences per scan component
};

// True when the bits from the reader's position to the end of the stream (end_rel, same base) are only
// the 1-padding of the last byte (fewer than 8 bits, all ones): no Huffman code consists of ones only,
// so real data never looks like this.
template <class Src>
BJ_HD bool at_padding(const BitReader<Src>& rd, uint32_t end_rel) {
    if (rd.rel >= end_rel) return true;
    uint32_t left = end_rel - rd.rel;
    if (left >= 8) return false;
    uint32_t ones = (1u << left) - 1u;
    return rd.bits_after(0, (int)left) == ones;
}

#define BJ_M_BASE 0
#define BJ_M_DCFIRST 1

// All positions below are 32-bit and relative to the stream start (rd.base): own_rel = first bit of
// the subsequence (0xFFFFFFFF: count nothing), stop_rel = its end, end_rel = end of the stream.
// `lut` is the scan's LUT blob; it is a separate argument (not a field of ScanCtx) so that the CUDA
// compiler can see when it points to shared memory and emit LDS instead of generic loads.

// ---- baseline / DC-first: counting pass ----------------------------------------------------------
// Decode from the reader's position with state (z, slot) until rd.rel >= stop_rel.  Blocks whose DC
// symbol starts at a position >= own_rel are counted and their DC differences summed.  Nothing is
// written.  FLAT loop: every iteration decodes exactly one symbol (DC or AC, chosen by a table
// select), so the 32 lanes of a warp stay converged although their blocks have different numbers of
// symbols; only the short DC / end-of-block bodies diverge.
template <int MODE, class Src>
BJ_HD void sync_run(BitReader<Src>& rd, int& z, int& slot, const ScanCtx& c, const uint32_t* lut, uint32_t own_rel,
                    uint32_t stop_rel, uint32_t end_rel, SubCount& cnt) {
    const int nslots = c.nslots;
    uint32_t tabs = c.tabs[slot];
    // the 1-padding of the last byte can only be met within the last 7 bits of the stream, i.e. in its last
    // subsequence: everywhere else the test below is one compare that never fires
    const uint32_t pad_from = (stop_rel + 8u > end_rel) ? (end_rel >= 7u ? end_rel - 7u : 0u) : 0xFFFFFFFFu;
    while (rd.rel < stop_rel) {
        const bool is_dc = (z == 0);
        if (BJ_UNLIKELY(rd.rel >= pad_from)) {
            if (is_dc && at_padding(rd, end_rel)) {
                rd.rel = end_rel;
                break;
            }
        }
        const uint32_t pk = rd.peek32();
        const uint32_t e = lut_lookup(lut + (is_dc ? (tabs & 0xFFFFu) : (tabs >> 16)), pk >> 16);
        int adv = ent_adv(e);
        if (is_dc) {
            if (rd.rel >= own_rel) {
                const int L = ent_len(e);
                const int t = L ? ent_sym(e) : 0;
                cnt.blocks++;
                const int diff = t ? take_extend(pk, L, t) : 0;
                const int k = c.slot_comp[slot];
                if (k == 0) cnt.dc[0] += diff;
                else if (k == 1) cnt.dc[1] += diff;
                else cnt.dc[2] += diff;
            }
            adv = (MODE == BJ_M_DCFIRST) ? 64 : 1;
        }
        rd.skip(ent_total(e));  // entries that are not a code consume 1 bit: any deterministic step will do
        z += adv;
        if (z >= 64) {
            z = 0;
            slot = (slot + 1 == nslots) ? 0 : slot + 1;
            tabs = c.tabs[slot];
        }
    }
}

// ---- baseline: writing pass ----------------------------------------------------------------------
// Sink: begin(), put(zigzag_index, value), commit(block_in_stream, slot) -- one whole block at a time.
// Returns BJ_ERR_* bits.  `blk` is the index (within the stream) of the first block this thread
// owns; on return it is one past the last block written.  If z != 0 on entry the open block belongs
// to the previous subsequence: it is decoded without being written.
// This loop is nested (per block: DC, AC symbols, commit) on purpose: the 24-instruction block flush
// then runs with all lanes of the warp converged, which measured faster on B200 than the flat form
// (2.8 vs 3.9 ms per 512 images) even though lanes wait for the block with the most symbols.
template <class Src, class Sink>
BJ_HD uint32_t base_write_run(BitReader<Src>& rd, int z, int slot, const ScanCtx& c, const uint32_t* lut, uint32_t stop_rel,
                              uint32_t end_rel, uint32_t& blk, uint32_t nblk_stream, int pred[3], Sink& sink) {
    // Single-exit loops only (errors are carried in `err`, never returned from inside a loop): the
    // compiler then reconverges the warp after every inner loop, which this nested form relies on.
    const int nslots = c.nslots;
    uint32_t err = 0;
    if (z != 0) {
        const uint32_t* const tab = lut + c.ac_tab[slot];
        while (z < 64) {
            uint32_t e = lut_lookup(tab, rd.peek16());
            if (ent_len(e) == 0) err |= BJ_ERR_BAD_CODE;
            if (rd.rel >= end_rel + 64) err |= BJ_ERR_OVERRUN;
            rd.skip(ent_total(e));
            z += err ? 64 : ent_adv(e);
        }
        slot = (slot + 1 == nslots) ? 0 : slot + 1;
    }
    // The 32 lanes of a warp walk their blocks in lock step, one block per round, and a round lasts as long as its
    // longest block.  Luma blocks carry three times the symbols of chroma blocks, so the rounds are kept in PHASE:
    // round k is for slot k mod nslots, a lane whose next block sits in another slot of the MCU idles until the
    // rotation reaches it (fewer than nslots rounds, once).  From then on every lane decodes the same kind of block in
    // every round: 4:2:0 content needs about a fifth fewer symbol iterations than with mixed rounds.
    int phase = 0;
    while (err == 0 && rd.rel < stop_rel && blk < nblk_stream) {
        const bool mine = (slot == phase);
        phase = (phase + 1 == nslots) ? 0 : phase + 1;
        if (!mine) continue;
        sink.begin();
        {
            const uint32_t pk = rd.peek32();
            uint32_t e = lut_lookup(lut + c.dc_tab[slot], pk >> 16);
            int L = ent_len(e), t = ent_sym(e);
            if (L == 0) { err |= BJ_ERR_BAD_CODE; t = 0; }
            const int diff = t ? take_extend(pk, L, t) : 0;
            int k = c.slot_comp[slot];
            int pv;
            if (k == 0) pv = (pred[0] += diff);
            else if (k == 1) pv = (pred[1] += diff);
            else pv = (pred[2] += diff);
            sink.put(0, (int16_t)pv);  // previous_dc is int16 (:735, :818-820)
            rd.skip(ent_total(e));
        }
        const uint32_t* const tab = lut + c.ac_tab[slot];
        int zz = 0;  // last coefficient written
        while (zz < 63) {
            const uint32_t pk = rd.peek32();
            const uint32_t e = lut_lookup(tab, pk >> 16);
            const int L = ent_len(e), tot = ent_total(e);
            const int s = tot - L;
            zz += ent_adv(e);  // zero run + 1 (EOB: jumps past 63, ZRL: 16 with no value)
            if (BJ_UNLIKELY(L == 0)) { err |= BJ_ERR_BAD_CODE; zz = 64; }
            if (s && zz < 64) sink.put(zz, (int16_t)take_extend(pk, L, s));
            rd.skip(tot);
        }
        if (rd.rel > end_rel + 7) err |= BJ_ERR_OVERRUN;
        if (err == 0) {
            sink.commit(blk, slot);
            blk++;
        }
        slot = (slot + 1 == nslots) ? 0 : slot + 1;
    }
    return err;
}

// ---- DC first: writing pass (one 16-bit store per block) -----------------------------------------
template <class Src, class Sink>
BJ_HD uint32_t dcfirst_write_run(BitReader<Src>& rd, int slot, const ScanCtx& c, const uint32_t* lut, uint32_t stop_rel,
                                 uint32_t end_rel, uint32_t& blk, uint32_t nblk_stream, int pred[3], Sink& sink) {
    while (rd.rel < stop_rel && blk < nblk_stream) {
        const uint32_t pk = rd.peek32();
        uint32_t e = lut_lookup(lut + c.dc_tab[slot], pk >> 16);
        int L = ent_len(e), t = ent_sym(e);
        if (L == 0) return BJ_ERR_BAD_CODE;
        int diff = extend(t ? take_bits(pk, L, t) : 0u, t);
        int k = c.slot_comp[slot];
        int pv;
        if (k == 0) pv = (pred[0] += diff);
        else if (k == 1) pv = (pred[1] += diff);
        else pv = (pred[2] += diff);
        rd.skip(ent_total(e));
        if (rd.rel > end_rel + 7) return BJ_ERR_OVERRUN;
        sink.store_dc(blk, slot, (int16_t)((uint32_t)(int32_t)(int16_t)pv << c.al));  // (:1029)
        blk++;
        slot = (slot + 1 == c.nslots) ? 0 : slot + 1;
    }
    return 0;
}

// ---- AC first (:1120-1256) -----------------------------------------------------------------------
// State: zig-zag index z in [ss, se].  A symbol either places a coefficient after a zero run, skips
// 16 zeros (ZRL), or ends the band of this block and of the next EOBRUN-1 blocks.  WRITE = false:
// count block advance only; WRITE = true: also store coefficients of symbols that start at or
// after own_rel (symbol-level ownership; the planes were zeroed before the first scan).
template <bool WRITE, class Src, class Sink>
BJ_HD uint32_t acfirst_run(BitReader<Src>& rd, int& z, const ScanCtx& c, const uint32_t* lut, uint32_t own_rel,
                           uint32_t stop_rel, uint32_t end_rel, uint32_t& blk, uint32_t nblk_stream, uint32_t& advance,
                           Sink& sink) {
    const uint32_t* tab = lut + c.ac_tab[0];
    const bool near_end = stop_rel + 8u > end_rel;  // see sync_run
    while (rd.rel < stop_rel) {
        if (WRITE && blk >= nblk_stream) break;
        if (near_end && end_rel - rd.rel < 8 && at_padding(rd, end_rel)) {
            rd.rel = end_rel;
            break;
        }
        const uint32_t pk = rd.peek32();
        uint32_t e = lut_lookup(tab, pk >> 16);
        int L = ent_len(e), rs = ent_sym(e);
        bool own = rd.rel >= own_rel;
        if (L == 0) {
            if (WRITE) return BJ_ERR_BAD_CODE;
            rd.skip(1);
            continue;
        }
        int r = rs >> 4, s = rs & 15;
        uint32_t adv = 0;
        if (s) {
            z += r;
            if (WRITE && own) {
                if (z > 63) return BJ_ERR_COEF_INDEX;
                sink.store(blk, z, (int16_t)((uint32_t)extend(take_bits(pk, L, s), s) << c.al));  // (:1225)
            }
            z++;
            rd.skip(L + s);
        } else if (r == 15) {
            z += 16;  // (:1142-1143)
            rd.skip(L);
        } else {
            uint32_t run = (1u << r) + (r ? take_bits(pk, L, r) : 0u);  // (:1144-1149)
            rd.skip(L + r);
            adv = run;
            z = c.ss;
        }
        if (z > c.se) {
            adv = 1;
            z = c.ss;
        }
        blk += adv;
        if (own) advance += adv;
    }
    return 0;
}

// ---- AC refinement (:1100-1115, :1183-1198, :1209-1232, :1258-1292) -------------------------------
// The number of correction bits that follow a symbol depends on which coefficients of the block are
// already non-zero, so a refinement stream cannot be entered at a guessed state: the bit parse is
// sequential.  What CAN be taken off the sequential path is everything but the parse itself.  The
// non-zero history of a block is a 64-bit mask (bit z = coefficient z is non-zero; known before the
// scan starts), and with it a symbol costs one table lookup plus a few bit operations: "skip r
// zero-history coefficients" is "find the (r+1)-th clear bit", the correction bits passed on the way
// are a population count.  So the stage runs in two passes:
//   parse (acrefine_block<false>, one lane per stream, masks staged by the whole warp): walks the
//         symbols touching no coefficient, and records for every block the bit position where its
//         data starts (bit 31 set: the block lies inside an end-of-band run);
//   apply (acrefine_block<true>, one thread per block): decodes the block again from that position
//         and performs the stores -- fully parallel.
// Correction is the reference's `coef |= bit << Al` on the two's-complement value (:1114), which is
// NOT the T.81 rule for negative coefficients; bit-exact parity with the reference requires it.
// T81 = true applies the T.81 rule instead (G.1.2.3, libjpeg-turbo's decode_mcu_AC_refine): a set bit adds
// +-(1 << Al) by the coefficient's sign when that bit of its magnitude is still clear (compat="libjpeg-turbo").
// Both rules keep every non-zero coefficient non-zero, so the non-zero masks and the parse are the same.
BJ_HD int popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
BJ_HD int ctz64(uint64_t x) {  // x != 0
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)x) - 1;
#else
    return __builtin_ctzll(x);
#endif
}
// position of the n-th (n >= 1) set bit of x, or -1
BJ_HD int nth_set64(uint64_t x, int n) {
    for (int i = 1; i < n; i++) x &= x - 1;
    return x ? ctz64(x) : -1;
}

#define BJ_ACR_IN_EOBRUN 0x80000000u  // flag in the per-block start position

// The correction bits of the non-zero coefficients in `passed` (bit i = coefficient base + i), in
// increasing zig-zag order (:1107-1115).
template <bool APPLY, bool T81 = false, class Src>
BJ_HD void acrefine_corrections(BitReader<Src>& rd, uint64_t passed, int base, int16_t* p, int al) {
    int n = popc64(passed);
    if (!APPLY) {
        rd.skip_long((uint32_t)n);
        return;
    }
    while (n > 0) {
        const int k = n < 32 ? n : 32;
        const uint32_t v = rd.peek32();
        for (int i = 0; i < k; i++) {
            const int zz = ctz64(passed);
            passed &= passed - 1;
            if constexpr (T81) {
                const int c = p[base + zz];
                if (((v << i) & 0x80000000u) && !(c & (1 << al))) p[base + zz] = (int16_t)(c >= 0 ? c + (1 << al) : c - (1 << al));
            } else {
                if ((v << i) & 0x80000000u) p[base + zz] = (int16_t)(p[base + zz] | (int16_t)(1 << al));
            }
        }
        rd.skip(k);
        n -= k;
    }
}

// One block of an AC refinement stream.  m = non-zero history of the block (all 64 positions),
// eob_run = blocks still covered by a running end-of-band run (0: the block starts with a symbol).
// APPLY = false only advances the reader; APPLY = true also updates the block at p.
template <bool APPLY, bool T81 = false, class Src>
BJ_HD uint32_t acrefine_block(BitReader<Src>& rd, const ScanCtx& c, const uint32_t* tab, uint32_t end_rel, uint64_t m,
                              uint32_t& eob_run, int16_t* p) {
    const int ss = c.ss, se = c.se, al = c.al;
    int z = ss;
    if (eob_run == 0) {
        while (z <= se) {
            if (rd.rel > end_rel + 7) return BJ_ERR_OVERRUN;
            const uint32_t pk = rd.peek32();
            const uint32_t e = lut_lookup(tab, pk >> 16);
            const int L = ent_len(e), rs = ent_sym(e);
            if (L == 0) return BJ_ERR_BAD_CODE;
            const int r = rs >> 4, s = rs & 15;
            if (s == 0 && r != 15) {  // EOBn (:1144-1149); EOB0 is a run of one block
                eob_run = (1u << r) + (r ? take_bits(pk, L, r) : 0u);
                rd.skip(L + r);
                break;
            }
            // skip r zero-history coefficients (16 for ZRL), refining the non-zero ones passed
            // (:1184-1193); with s != 0 go on to the next zero-history position, where the new
            // coefficient lands (:1211-1215).  Its value bits come right after the code (:1202).
            int newval = 0;
            if (s) newval = extend(take_bits(pk, L, s), s);
            rd.skip(L + s);
            const uint64_t rest = m >> z;
            const uint64_t zeros = ~rest & (~0ull >> z);
            const int idx = nth_set64(zeros, s ? r + 1 : 16);
            if (idx < 0) return BJ_ERR_COEF_INDEX;
            acrefine_corrections<APPLY, T81>(rd, rest & ((1ull << idx) - 1ull), z, p, al);
            if (APPLY && s) p[z + idx] = (int16_t)((uint32_t)newval << al);  // (:1225)
            z += idx + 1;
        }
        if (z > se) return 0;
    }
    // end-of-band run: the rest of this band (and the whole band of the blocks that follow inside the
    // run) only carries correction bits for its non-zero coefficients (:1258-1292)
    const uint64_t band = (~0ull << z) & (~0ull >> (63 - se));
    acrefine_corrections<APPLY, T81>(rd, m & band, 0, p, al);
    eob_run--;
    return rd.rel > end_rel + 7 ? BJ_ERR_OVERRUN : 0u;
}

// ---- the sequential parse, made as short as a single lane allows -----------------------------------
// Per block the warp prepares a small table from the non-zero mask: zpos[k] = zig-zag position of the
// k-th zero-history coefficient at or after Ss (0xFF: none), and the number of non-zero coefficients
// in the band.  With j = zero-history coefficients consumed so far, a symbol with run r lands on
// zpos[j + r], and the correction bits passed since the previous landing are the non-zero
// coefficients in between: (zpos[t] - t) - (previous zpos - previous t).  One table lookup for the
// code, one for the landing, a handful of integer operations -- no loop over coefficients.
#define BJ_ACR_TAB_STRIDE 100  // bytes per block table; 25 words: conflict-free when lanes fill theirs
#define BJ_ACR_TAB_NZ 80       // index of the band's non-zero count

BJ_HD void acrefine_build_table(uint64_t m, int ss, int se, uint8_t* t) {
    uint64_t zm = ~m & (~0ull << ss);
    int k = 0;
    while (zm) {
        t[k++] = (uint8_t)ctz64(zm);
        zm &= zm - 1;
    }
    for (; k < BJ_ACR_TAB_NZ; k++) t[k] = 0xFF;
    t[BJ_ACR_TAB_NZ] = (uint8_t)popc64(m & (~0ull << ss) & (~0ull >> (63 - se)));
}

// ---- the sequential parse over a PRE-DECODED WINDOW -----------------------------------------------------
// What makes the parse slow is not the work but the length of the dependency chain per symbol (one lane, every
// instruction at full latency).  Everything that depends only on the BIT POSITION is therefore taken off the chain:
// the warp decodes the Huffman symbol that WOULD start at each of the next BJ_ACR_WIN_BITS bit positions, all in
// parallel, into a shared-memory window (acrefine_predecode: code length + sign bit, run, EOBn with its run count).
// The chain that is left per symbol is: window entry at the current position -> landing position from the block's
// table (depends on the run) -> next position.  Two dependent shared-memory loads and a handful of integer
// operations instead of a funnel shift, a two-level LUT walk, field extraction and the refill logic.
#ifndef BJ_ACR_WIN_BITS
#define BJ_ACR_WIN_BITS 8192
#endif
// A block that starts inside [window start, window start + BJ_ACR_WIN_BITS - BJ_ACR_WIN_SLACK] has all its symbol
// starts inside the window: at most 64 symbols (each lands on a new coefficient) of at most 16 + 1 bits, 63
// correction bits, one EOBn of 16 + 14 bits.
#define BJ_ACR_WIN_SLACK 1280
#define BJ_ACR_E_EOB 0x1000u   // entry: end of band (bits 16..31: blocks the run still covers AFTER this one)
#define BJ_ACR_E_BAD 0x2000u   // entry: not a code, or a size other than 0 / 1 (ends the block, flags the stream)

// Window entry for the symbol that starts at absolute bit `abs_bit`: bits 0..7 = bits consumed by code + sign (or
// + EOBRUN bits), bits 8..11 = run.
template <class Src>
BJ_HD uint32_t acrefine_predecode(const Src& src, uint64_t abs_bit, const uint32_t* tab) {
    const uint32_t w = (uint32_t)(abs_bit >> 5);
    const uint32_t pk = funnel_left(src.word(w), src.word(w + 1), (int)(abs_bit & 31));
    const uint32_t e = lut_lookup(tab, pk >> 16);
    const int L = ent_len(e), rs = ent_sym(e);
    const int r = rs >> 4, s = rs & 15;
    if (L == 0 || s > 1) return 1u | BJ_ACR_E_EOB | BJ_ACR_E_BAD;   // consumes one bit, ends the block like EOB0
    if (s == 0 && r != 15) {                                         // EOBn (:1144-1149); EOB0 is a run of one block
        const uint32_t run = (1u << r) + (r ? take_bits(pk, L, r) : 0u) - 1u;
        return (uint32_t)(L + r) | BJ_ACR_E_EOB | (run << 16);
    }
    return (uint32_t)(L + s) | ((uint32_t)r << 8);
}

// Parse blocks [i0, nb) of a chunk (tables at tabs + i * BJ_ACR_TAB_STRIDE) from bit position `pos` (relative to the
// stream start) while they start at or before win_limit; pre[k] = entry of position win_base + k.  blkpos[i]
// receives where block i starts (| BJ_ACR_IN_EOBRUN).  Returns the index of the first block NOT parsed; err != 0
// stops the stream.  Written for the shortest dependency chain: no early exits inside a block, problems are
// collected in sticky flags and looked at once per block; a run past the last zero-history coefficient (table
// entry 0xFF >= se) ends the block.
BJ_HD int acrefine_parse_window(const uint32_t* pre, uint32_t win_base, uint32_t win_limit, const ScanCtx& c, uint32_t end_rel,
                                const uint8_t* tabs, int i0, int nb, uint32_t& pos, uint32_t& eob_run, uint32_t* blkpos,
                                uint32_t& err) {
    const int ss = c.ss, se = c.se;
    uint32_t bad_code = 0, bad_index = 0;
    int i = i0;
    // the chain runs on p = position inside the window (an index into pre[]); pos = win_base + p
    if (win_base > end_rel + 7u) {   // the window itself starts past the end of the stream
        err = BJ_ERR_OVERRUN;
        return i0;
    }
    uint32_t p = pos - win_base;
    const uint32_t p_limit = win_limit - win_base, p_end = end_rel + 7u - win_base;
    for (; i < nb; i++) {
        if (p > p_limit) break;
        const uint8_t* t = tabs + i * BJ_ACR_TAB_STRIDE;
        if (p > p_end) {
            err = BJ_ERR_OVERRUN;
            pos = win_base + p;
            return i;
        }
        if (eob_run) {
            blkpos[i] = (win_base + p) | BJ_ACR_IN_EOBRUN;
            p += t[BJ_ACR_TAB_NZ];
            eob_run--;
            continue;
        }
        blkpos[i] = win_base + p;
        int j = 0;     // zero-history coefficients consumed
        int cd = ss;   // ss + non-zero coefficients refined so far
        for (;;) {
            // the chain: window entry -> run -> table entry -> next position.  Nothing else may sit on it: a run past
            // the last zero-history coefficient (table entry 0xFF) makes p meaningless, but it also ends the block
            // (0xFF >= se) and is reported right after it.
            const uint32_t e = pre[p];
            if (e & BJ_ACR_E_EOB) {
                bad_code |= e & BJ_ACR_E_BAD;
                eob_run = e >> 16;
                p += (e & 0xFFu) + (uint32_t)((int)t[BJ_ACR_TAB_NZ] - (cd - ss));
                break;
            }
            const int tt = j + (int)byte_of(e, 1);          // ZRL: the 16th zero from here (run 15)
            const int zp = t[tt];
            p += (uint32_t)((int)byte_of(e, 0) - tt - cd + zp);  // code + sign bits, then one correction bit per non-zero passed
            cd = zp - tt;
            j = tt + 1;
            if (zp >= se) {
                bad_index |= (zp == 0xFF) ? 1u : 0u;
                break;
            }
        }
        if (bad_code | bad_index) {
            err = bad_code ? BJ_ERR_BAD_CODE : BJ_ERR_COEF_INDEX;
            pos = win_base + p;
            return i;
        }
    }
    pos = win_base + p;
    return i;
}

}  // namespace bj
