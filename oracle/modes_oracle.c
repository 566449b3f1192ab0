/*
 * modes_oracle.c — CPU restatement of readsb's 2.4 MSPS Mode-S demodulator (TEST INFRASTRUCTURE).
 *
 * See modes_oracle.h for the role of this file and how it is pinned against the reference.
 * Written from the behaviour of the reference (file:line cited per function), not from its text:
 * the bit slicer uses the closed form  u = phase + 12*k, sample = j + 19 + u/5, correlator = u%5
 * instead of the reference's unrolled slice_byte switch, the error tables are a direct
 * syndrome scan, and the ICAO filter is a plain two-generation set.
 *
 * Build:  gcc -O2 -std=c11 -ffp-contract=off -fPIC -shared modes_oracle.c -o libmodes_oracle.so -lm
 *         (-ffp-contract=off matters: the LUT arithmetic must round mul and add separately,
 *          like the reference built with plain -O2 on x86-64.)
 */
#include "modes_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define TRAIL B200_TRAILING_SAMPLES
#ifndef M_SQRT2
#define M_SQRT2 1.41421356237309504880 /* math.h value (hidden by -std=c11) */
#endif

/* ------------------------------------------------------------------ convert.c:35-62 */
static uint16_t g_lut[65536];
static int g_lut_ready;

static void build_lut(void) {
    if (g_lut_ready) return;
    for (int i = 0; i < 256; i++) {
        for (int q = 0; q < 256; q++) {
            float fi = (float)((i - 127.5) / 127.5); /* double divide, then narrowed (convert.c:49) */
            float fq = (float)((q - 127.5) / 127.5);
            float magsq = fi * fi + fq * fq;          /* float mul, float add, no contraction */
            if (magsq > 1) magsq = 1;
            float mag = sqrtf(magsq);
            /* index: the reference reads each I,Q byte pair as a little-endian uint16 (convert.c:70,78)
             * into a table filled at [i*256+q]; the table is symmetric in i<->q so either order
             * gives the same value. */
            g_lut[i * 256 + q] = (uint16_t)(mag * 65535.0f + 0.5f);
        }
    }
    g_lut_ready = 1;
}

void oracle_uc8_lut(uint16_t *out) {
    build_lut();
    memcpy(out, g_lut, sizeof(g_lut));
}

/* ------------------------------------------------------------------ convert.c:64-108 */
void oracle_convert_uc8(const uint8_t *iq, uint16_t *mag, unsigned n, uint64_t *sum_level, uint64_t *sum_power) {
    build_lut();
    uint64_t sl = 0, sp = 0;
    for (unsigned k = 0; k < n; k++) {
        /* little-endian uint16 read of (I,Q): index = I + 256*Q */
        unsigned idx = (unsigned)iq[2 * k] | ((unsigned)iq[2 * k + 1] << 8);
        uint16_t m = g_lut[idx];
        mag[k] = m;
        sl += m;
        sp += (uint64_t)((uint32_t)m * (uint32_t)m);
    }
    if (sum_level) *sum_level = sl;
    if (sum_power) *sum_power = sp;
}

/* ------------------------------------------------------------------ crc.c:42-82 */
#define POLY 0xfff409u
static uint32_t g_crc_tab[256];
static uint32_t g_bit_syn[112]; /* syndrome of a single set bit i of a 112-bit frame (crc.c:59-64) */
static int g_crc_ready;

static void build_crc_tab(void) {
    if (g_crc_tab[1]) return;   /* entry 1 is POLY once built */
    for (int i = 0; i < 256; i++) {
        uint32_t c = (uint32_t)i << 16;
        for (int j = 0; j < 8; j++) c = (c & 0x800000) ? ((c << 1) ^ POLY) : (c << 1);
        g_crc_tab[i] = c & 0xffffff;
    }
}

/* callable first thing in a process: builds the table it reads */
uint32_t oracle_crc24(const uint8_t *msg, int bits) {
    build_crc_tab();
    int n = bits / 8;
    uint32_t rem = 0;
    for (int i = 0; i < n - 3; i++)
        rem = ((rem << 8) ^ g_crc_tab[msg[i] ^ ((rem >> 16) & 0xff)]) & 0xffffff;
    return rem ^ ((uint32_t)msg[n - 3] << 16) ^ ((uint32_t)msg[n - 2] << 8) ^ msg[n - 1];
}

static void build_crc(void) {
    if (g_crc_ready) return;
    build_crc_tab();
    uint8_t m[14];
    for (int i = 0; i < 112; i++) {
        memset(m, 0, sizeof m);
        m[i >> 3] = (uint8_t)(1u << (7 - (i & 7)));
        g_bit_syn[i] = oracle_crc24(m, 112);
    }
    g_crc_ready = 1;
}

/* crc.c:180-406 with max_correct = 1: the table holds the syndromes of single-bit errors at message
 * bits 5..bits-1 (DF bits are never corrected, crc.c:210-211); a short frame's bit i has the
 * syndrome of long-frame bit i+56 (offset = 112-bits).  All 107 / 51 syndromes are distinct, so
 * the bsearch is equivalent to this scan. */
int oracle_crc_diagnose1(uint32_t syndrome, int bits) {
    build_crc();
    if (syndrome == 0) return -1;
    int off = 112 - bits;
    for (int b = 5; b < bits; b++)
        if (g_bit_syn[b + off] == syndrome) return b;
    return -2;
}

/* crc.c:180-378 with max_correct = 2, max_detect = 4 (modesChecksumInit's `default:` case, i.e. --aggressive,
 * readsb.c:1535-1537).  PREPARATION for a later round: nothing on the demodulator path of this oracle uses it yet (the
 * library refuses nfix_crc = 2), but the table is the part that has to be exactly the reference's, so it is restated and
 * pinned now.  The reference enumerates every 1- and 2-bit error pattern over message bits 5..bits-1, sorts by syndrome,
 * drops every syndrome that occurs more than once, then drops every entry whose syndrome is also the syndrome of some 3- or
 * 4-bit pattern (flagCollisions).  The same set, built with a bit per syndrome instead of sorting and searching:
 *   keep(s) <=> exactly one pattern of <= 2 bits has syndrome s, and no pattern of 3 or 4 bits has it. */
typedef struct { uint32_t syndrome; int8_t b0, b1; } err2;
static err2 *g_tab2[2]; static int g_ntab2[2];        /* [0] 56-bit, [1] 112-bit, sorted by syndrome */

static int err2_cmp(const void *a, const void *b) { return (int)((const err2 *)a)->syndrome - (int)((const err2 *)b)->syndrome; }

static void build_tab2(int which) {
    if (g_tab2[which]) return;
    build_crc();
    const int bits = which ? 112 : 56, off = 112 - bits, n = bits - 5;
    const uint32_t *syn = &g_bit_syn[5 + off];                      /* syn[i] = syndrome of message bit 5 + i */
    uint8_t *seen12 = calloc(1 << 21, 1), *dup12 = calloc(1 << 21, 1), *seen34 = calloc(1 << 21, 1);
#define BIT(a, x) ((a)[(x) >> 3] >> ((x) & 7) & 1)
#define SET(a, x) ((a)[(x) >> 3] |= (uint8_t)(1u << ((x) & 7)))
    for (int i = 0; i < n; i++) {
        uint32_t s1 = syn[i];
        if (BIT(seen12, s1)) SET(dup12, s1); else SET(seen12, s1);
        for (int j = i + 1; j < n; j++) {
            uint32_t s2 = s1 ^ syn[j];
            if (BIT(seen12, s2)) SET(dup12, s2); else SET(seen12, s2);
            for (int k = j + 1; k < n; k++) {
                uint32_t s3 = s2 ^ syn[k];
                SET(seen34, s3);
                for (int l = k + 1; l < n; l++) SET(seen34, s3 ^ syn[l]);
            }
        }
    }
    err2 *t = malloc(sizeof(err2) * (size_t)(n + n * (n - 1) / 2));
    int m = 0;
    for (int i = 0; i < n; i++) {
        uint32_t s1 = syn[i];
        if (!BIT(dup12, s1) && !BIT(seen34, s1)) { t[m].syndrome = s1; t[m].b0 = (int8_t)(5 + i); t[m].b1 = -1; m++; }
        for (int j = i + 1; j < n; j++) {
            uint32_t s2 = s1 ^ syn[j];
            if (!BIT(dup12, s2) && !BIT(seen34, s2)) { t[m].syndrome = s2; t[m].b0 = (int8_t)(5 + i); t[m].b1 = (int8_t)(5 + j); m++; }
        }
    }
#undef BIT
#undef SET
    free(seen12); free(dup12); free(seen34);
    qsort(t, (size_t)m, sizeof(err2), err2_cmp);
    g_tab2[which] = t; g_ntab2[which] = m;
}

/* modesChecksumDiagnose (crc.c:383-406) for --aggressive: returns the number of errors (0 for syndrome 0, 1 or 2 with the
 * bit positions in *b0 / *b1, ascending), or -2 when the syndrome is not in the table. */
int oracle_crc_diagnose2(uint32_t syndrome, int bits, int *b0, int *b1) {
    *b0 = *b1 = -1;
    if (syndrome == 0) return 0;
    const int which = bits == 112;
    build_tab2(which);
    err2 key; key.syndrome = syndrome;
    const err2 *e = bsearch(&key, g_tab2[which], (size_t)g_ntab2[which], sizeof(err2), err2_cmp);
    if (!e) return -2;
    *b0 = e->b0; *b1 = e->b1;
    return e->b1 >= 0 ? 2 : 1;
}

/* Entries of the table and a digest over (syndrome, errors, bits) of every entry, for pinning against the reference. */
int oracle_crc_table2_digest(int bits, uint64_t *digest) {
    const int which = bits == 112;
    build_tab2(which);
    uint64_t h = 1469598103934665603ull;
    for (int i = 0; i < g_ntab2[which]; i++) {
        const err2 *e = &g_tab2[which][i];
        const uint64_t v = ((uint64_t)e->syndrome << 16) | ((uint64_t)(uint8_t)e->b0 << 8) | (uint8_t)e->b1;
        h = (h ^ v) * 1099511628211ull;
    }
    *digest = h;
    return g_ntab2[which];
}

/* ------------------------------------------------------------------ icao_filter.c semantics
 * Two generations; Test looks in both (icao_filter.c:132-154), Add goes to the active one
 * (:112-130), Expire clears the other one and makes it active (:96-110).  The reference's hash LAYOUT is
 * unobservable, its table SIZE is not: icaoFilterAdd doubles both tables once the active one holds more than
 * buckets / 3 addresses (:126-128) and icaoFilterResize re-inserts the active generation only (:66-92) - the older
 * generation is forgotten at that moment (the 86th, 171st, 342nd ... new address of a generation, starting from
 * 2^8 buckets); icaoFilterExpire halves the tables first when the active generation holds fewer than buckets / 9
 * (:97-99).  So the observable state is two sets plus `bits`; the sets themselves are growable open-addressed
 * sets of this file's own design. */
typedef struct { uint32_t *slot; uint32_t cap, n; } aset;

static void aset_init(aset *s) { s->cap = 1024; s->n = 0; s->slot = malloc(s->cap * 4); memset(s->slot, 0xff, s->cap * 4); }
static void aset_clear(aset *s) { memset(s->slot, 0xff, s->cap * 4); s->n = 0; }
static uint32_t aset_h(uint32_t a) { a *= 0x9E3779B1u; return a ^ (a >> 15); }
static int aset_has(const aset *s, uint32_t a) {
    uint32_t h = aset_h(a) & (s->cap - 1);
    while (s->slot[h] != 0xffffffffu) { if (s->slot[h] == a) return 1; h = (h + 1) & (s->cap - 1); }
    return 0;
}
static void aset_add(aset *s, uint32_t a) {
    if (aset_has(s, a)) return;
    if ((s->n + 1) * 2 > s->cap) {
        aset t = { malloc(s->cap * 2 * 4), s->cap * 2, 0 };
        memset(t.slot, 0xff, t.cap * 4);
        for (uint32_t i = 0; i < s->cap; i++) if (s->slot[i] != 0xffffffffu) {
            uint32_t h = aset_h(s->slot[i]) & (t.cap - 1);
            while (t.slot[h] != 0xffffffffu) h = (h + 1) & (t.cap - 1);
            t.slot[h] = s->slot[i]; t.n++;
        }
        free(s->slot); *s = t;
    }
    uint32_t h = aset_h(a) & (s->cap - 1);
    while (s->slot[h] != 0xffffffffu) h = (h + 1) & (s->cap - 1);
    s->slot[h] = a; s->n++;
}

struct oracle_ctx {
    int thr, nfix, fixdf, ttl_ms;
    uint32_t long_set, short_set;     /* demod_2400.c:98-128 */
    aset gen[2]; int active;
    int filter_bits;                  /* icao_filter.c:30,45-46: log2 of the reference's bucket count, 8..20 */
    int64_t next_flip; int flip_armed;
    /* stream state for oracle_run_stream_uc8 */
    uint16_t halo[TRAIL]; int halo_valid;
    uint32_t buffer_seq;
    b200_demod_stats st;
};

void oracle_icao_add(oracle_ctx *o, uint32_t a) {
    aset *act = &o->gen[o->active];
    aset_add(act, a);                                                  /* icao_filter.c:112-124 (`occupied` = size of the active set) */
    if (act->n > (1u << o->filter_bits) / 3 && o->filter_bits < 20) {  /* :126-128 -> icaoFilterResize :66-92 */
        o->filter_bits++;
        aset_clear(&o->gen[o->active ^ 1]);                            /* only the active generation is re-inserted */
    }
}
int oracle_icao_test(const oracle_ctx *o, uint32_t a) { return aset_has(&o->gen[0], a) || aset_has(&o->gen[1], a); }
void oracle_icao_expire(oracle_ctx *o) {
    if (o->gen[o->active].n < (1u << o->filter_bits) / 9 && o->filter_bits > 8) o->filter_bits--;   /* icao_filter.c:97-99 */
    o->active ^= 1; aset_clear(&o->gen[o->active]); o->st.icao_flips++;
}

/* Modes.preambleThreshold is re-read for every buffer (demod_2400.c:334-338): the caller applies the reference's
 * "at least PREAMBLE_THRESHOLD_PIZERO (75) while samples were dropped recently" rule between buffers. */
void oracle_set_preamble_threshold(oracle_ctx *o, int thr) { if (thr > 0) o->thr = thr; }

oracle_ctx *oracle_create(int thr, int nfix, int fixdf, int ttl_ms) {
    build_lut(); build_crc();
    oracle_ctx *o = calloc(1, sizeof *o);
    o->thr = thr ? thr : B200_PREAMBLE_THRESHOLD_DEFAULT;
    o->nfix = nfix ? 1 : 0; o->fixdf = fixdf ? 1 : 0;
    o->ttl_ms = ttl_ms == 0 ? B200_ICAO_TTL_MS : ttl_ms;
    /* demod_2400.c:112-127: DFs understood directly, plus every DF one bit away from 17 when
     * DF repair is on (generate_damage_set(17,1) = {17,16,19,21,25,1}). */
    o->short_set = (1u << 0) | (1u << 4) | (1u << 5) | (1u << 11);
    o->long_set = (1u << 16) | (1u << 17) | (1u << 18) | (1u << 20) | (1u << 21);
    if (o->fixdf && o->nfix) {
        o->long_set |= 1u << 17;
        for (int b = 0; b < 5; b++) o->long_set |= 1u << (17 ^ (1 << b));
    }
    aset_init(&o->gen[0]); aset_init(&o->gen[1]);
    o->filter_bits = 8;               /* icao_filter.c:45,50 MINBITS */
    return o;
}

void oracle_destroy(oracle_ctx *o) { if (!o) return; free(o->gen[0].slot); free(o->gen[1].slot); free(o); }
void oracle_get_stats(const oracle_ctx *o, b200_demod_stats *out) { *out = o->st; }

/* ------------------------------------------------------------------ demod_2400.c:74-93, 133-213
 * Correlator u%5 applied at sample j+19+u/5 for u = try_phase + 12*bit. */
static inline int slice_bit(const uint16_t *m, int row) {
    switch (row) {
        case 0: return 18 * m[0] - 15 * m[1] - 3 * m[2] > 0;
        case 1: return 14 * m[0] - 5 * m[1] - 9 * m[2] > 0;
        case 2: return 16 * m[0] + 5 * m[1] - 20 * m[2] > 0;
        case 3: return 7 * m[0] + 11 * m[1] - 18 * m[2] > 0;
        default: return 4 * m[0] + 15 * m[1] - 20 * m[2] + m[3] > 0;
    }
}

static void slice_bytes(const uint16_t *pa, int phase, int first_byte, int nbytes, uint8_t *msg) {
    for (int by = first_byte; by < nbytes; by++) {
        unsigned v = 0;
        for (int b = 0; b < 8; b++) {
            int u = phase + 12 * (by * 8 + b);
            v = (v << 1) | (unsigned)slice_bit(pa + 19 + u / 5, u % 5);
        }
        msg[by] = (uint8_t)v;
    }
}

static inline uint32_t aa_field(const uint8_t *m) { return ((uint32_t)m[1] << 16) | ((uint32_t)m[2] << 8) | m[3]; }

/* What one sliced phase looks like before the ICAO filter is consulted. */
typedef struct {
    uint8_t msg[14];
    int df;          /* DF as sliced */
    int nbytes;      /* bytes sliced (7/14) */
    int dfrepair;    /* fixDF17msgtype would succeed (mode_s.c:276-301) */
    uint32_t crc;    /* syndrome over modesMessageLenByType(df) bits of the unrepaired frame */
    int fixbit;      /* -1 crc==0 (or IID-only for DF11), >=5 correctable bit, -2 uncorrectable */
} sliced;

/* mode_s.c:309-419.  Returns the score; *addr_out = address that was looked up (for diagnostics). */
static int score_sliced(const oracle_ctx *o, const sliced *s) {
    const uint8_t *msg = s->msg;
    if (s->dfrepair) /* mode_s.c:319-329 */
        return oracle_icao_test(o, aa_field(msg)) ? 900 : 700;
    int df = s->df;
    /* validbits < msgbits cannot happen: nbytes was chosen from the DF. mode_s.c:336-338: */
    static const uint8_t z[7] = {0};
    if (!memcmp(msg, z, 7)) return -2;
    uint32_t crc = s->crc;
    switch (df) {
        case 0: case 4: case 5: case 16: case 20: case 21:
            return oracle_icao_test(o, crc) ? 1000 : -1;
        case 11: {
            uint32_t addr = aa_field(msg);
            if (crc & 0xffff80) {
                if (s->fixbit < 5) return -2;                       /* no table entry (or nfix=0) */
                if (s->fixbit >= 8 && s->fixbit <= 31) addr ^= 1u << (31 - s->fixbit); /* mode_s.c:230-245 */
                return oracle_icao_test(o, addr) ? 800 : -1;
            }
            if ((crc & 0x7f) == 0) return oracle_icao_test(o, addr) ? 1600 : 750;
            return oracle_icao_test(o, addr) ? 1000 : -1;
        }
        case 17: case 18: {
            if (s->fixbit == -2) return -2;
            uint32_t addr = aa_field(msg);
            int e = s->fixbit >= 5 ? 1 : 0;
            if (e && s->fixbit >= 8 && s->fixbit <= 31) addr ^= 1u << (31 - s->fixbit);
            return oracle_icao_test(o, addr) ? 1800 / (e + 1) : 1400 / (e + 1);
        }
        default:
            return -2;
    }
}

/* demod_2400.c:215-258 up to the score: slice, DF gate, CRC work that does not depend on the filter. */
static int slice_phase(const oracle_ctx *o, const uint16_t *pa, int phase, sliced *s) {
    slice_bytes(pa, phase, 0, 1, s->msg);
    int df = s->msg[0] >> 3;
    s->df = df;
    if (o->long_set & (1u << df)) s->nbytes = 14;
    else if (o->short_set & (1u << df)) s->nbytes = 7;
    else return 0; /* score -2 without slicing further */
    slice_bytes(pa, phase, 1, s->nbytes, s->msg);
    memset(s->msg + s->nbytes, 0, 14 - s->nbytes);
    s->dfrepair = 0;
    if (s->nbytes == 14 && o->fixdf && o->nfix && (df == 1 || df == 25 || df == 21 || df == 19 || df == 16)) {
        uint8_t t[14];
        memcpy(t, s->msg, 14);
        t[0] = (uint8_t)((t[0] & 7) | (17 << 3));
        if (oracle_crc24(t, 112) == 0) s->dfrepair = 1;
    }
    int bits = (df & 0x10) ? 112 : 56; /* mode_s.h:124 */
    s->crc = oracle_crc24(s->msg, bits);
    s->fixbit = -2;
    if (df == 11) {
        if (!(s->crc & 0xffff80)) s->fixbit = -1;
        else if (o->nfix) s->fixbit = oracle_crc_diagnose1(s->crc, bits);
    } else if (df == 17 || df == 18) {
        if (s->crc == 0) s->fixbit = -1;
        else if (o->nfix) s->fixbit = oracle_crc_diagnose1(s->crc, bits);
    }
    return 1;
}

/* ------------------------------------------------------------------ demod_2400.c:264-482 */
int oracle_demodulate2400(oracle_ctx *o, const uint16_t *m, unsigned mlen, int64_t sample_ts,
                          uint64_t sum_level, uint64_t sum_power,
                          b200_frame *out, unsigned cap, unsigned *n_out, b200_buffer_result *res) {
    b200_demod_stats *st = &o->st;
    const b200_demod_stats before = *st;        /* the buffer result reports what this call added to the counters */
    uint64_t sum_sig = 0;
    unsigned nfr = 0;
    int overflow = 0;
    int64_t now_ms = sample_ts / 12000; /* synthetic clock: buffer start (demod_2400.c:283-285) */

    for (unsigned j = 0; j < mlen; j++) {
        const uint16_t *pa = m + j;
        /* pre-check, demod_2400.c:311-320 (the reference's unroll tests every position) */
        if (!(pa[1] > pa[7] && pa[12] > pa[14] && pa[12] > pa[15])) continue;
        /* demod_2400.c:330-340 (samples_dropped never set on this path) */
        int32_t base_noise = pa[5] + pa[8] + pa[16] + pa[17] + pa[18];
        int32_t ref_level = (int32_t)((uint32_t)base_noise * (uint32_t)o->thr) >> 5;
        int32_t d23 = pa[2] - pa[3], s14 = pa[1] + pa[4], d1011 = pa[10] - pa[11];
        int32_t common = s14 - d23 + pa[9] + pa[12];
        int tryp[5], ntry = 0;
        if (common - d1011 >= ref_level) { tryp[ntry++] = 4; tryp[ntry++] = 5; }
        if (common + d1011 >= ref_level) { tryp[ntry++] = 6; tryp[ntry++] = 7; }
        if (s14 + 2 * d23 + d1011 + pa[12] >= ref_level) tryp[ntry++] = 8;
        if (!ntry) continue;

        int bestscore = -42, bestphase = 0;
        sliced best, cur;
        memset(&best, 0, sizeof best);
        for (int t = 0; t < ntry; t++) {
            st->demod_preamblePhase[tryp[t] - 4]++;
            int score = -2;
            if (slice_phase(o, pa, tryp[t], &cur)) score = score_sliced(o, &cur);
            if (score > bestscore) { /* strictly greater: earliest phase wins ties (demod_2400.c:243) */
                bestscore = score;
                if (score > -2) { best = cur; bestphase = tryp[t]; }
            }
        }
        st->demod_preambles++;
        if (bestscore < 0) {
            if (bestscore == -1) st->demod_rejected_unknown_icao++; else st->demod_rejected_bad++;
            continue;
        }

        /* accept part of decodeModesMessage, mode_s.c:443-596 + :766-779 */
        int msgtype = best.df, corrected = 0, fix_bit = -1;
        uint8_t msg[14];
        memcpy(msg, best.msg, 14);
        if (best.dfrepair) {
            fix_bit = 0; /* which DF bit differs from 17 */
            int x = best.df ^ 17;
            while (!((x << fix_bit) & 0x10)) fix_bit++;
            msg[0] = (uint8_t)((msg[0] & 7) | (17 << 3));
            msgtype = 17; corrected = 1;
        }
        int msgbits = (msgtype & 0x10) ? 112 : 56;
        uint32_t crc = best.dfrepair ? 0 : best.crc; /* mode_s.c:466 recomputed after repair */
        uint32_t addr;
        int result = 0, add_to_filter = 0;
        switch (msgtype) {
            case 0: case 4: case 5: case 16: case 20: case 21:
                addr = crc;
                if (!oracle_icao_test(o, crc)) result = -1;
                break;
            case 11:
                if (crc & 0xffff80) {
                    if (best.fixbit < 5) { result = -2; addr = 0; break; }
                    corrected = 1; fix_bit = best.fixbit;
                    msg[fix_bit >> 3] ^= (uint8_t)(1u << (7 - (fix_bit & 7)));
                    addr = aa_field(msg);
                    if (!oracle_icao_test(o, addr)) result = -1;
                } else {
                    addr = aa_field(msg);
                    if ((crc & 0x7f) == 0) add_to_filter = 1; /* IID == 0, no corrected bits */
                }
                break;
            case 17: case 18:
                addr = aa_field(msg);
                if (crc != 0) {
                    if (best.fixbit < 5) { result = -2; break; }
                    uint32_t addr1 = addr;
                    corrected = 1; fix_bit = best.fixbit;
                    msg[fix_bit >> 3] ^= (uint8_t)(1u << (7 - (fix_bit & 7)));
                    addr = aa_field(msg);
                    if (addr1 != addr && !oracle_icao_test(o, addr)) result = -1;
                } else if (msgtype == 17 && !corrected) {
                    add_to_filter = 1;
                }
                break;
            default:
                result = -2; addr = 0;
        }
        if (result < 0) {
            if (result == -1) st->demod_rejected_unknown_icao++; else st->demod_rejected_bad++;
            continue; /* no skip, demod_2400.c:422-428 */
        }
        if (add_to_filter) oracle_icao_add(o, addr);
        st->demod_accepted[corrected]++;
        st->demod_bestPhase[bestphase - 4]++;

        /* demod_2400.c:399,436-457: msglen comes from the DF as sliced (score restored byte 0) */
        int msglen = (best.df & 0x10) ? 112 : 56;
        int signal_len = msglen * 12 / 5;
        uint64_t sp = 0;
        for (int k = 0; k < signal_len; k++) { uint32_t v = pa[19 + k]; sp += (uint64_t)(v * v); }
        sum_sig += sp;
        st->signal_power_count += (uint64_t)signal_len;
        st->sum_signal_power += sp;
        double level = (double)sp / 65535.0 / 65535.0 / signal_len;
        if (level > st->peak_signal_power) st->peak_signal_power = level;
        if (level > 0.50119) st->strong_signal_count++;

        int64_t ts = sample_ts + (int64_t)j * 5 + (8 + 56) * 12 + bestphase; /* demod_2400.c:406 */
        now_ms = sample_ts / 12000 + (ts - sample_ts) / 12000;             /* :409-414 */
        if (*n_out < cap) {
            b200_frame *f = &out[(*n_out)++];
            memset(f, 0, sizeof *f);
            f->timestamp = ts; f->sigpow_sum = sp; f->j = j; f->crc = crc; f->addr = addr;
            f->score = bestscore; f->buffer_seq = o->buffer_seq; f->signal_len = (uint16_t)signal_len;
            f->phase = (uint8_t)bestphase; f->msgtype = (uint8_t)msgtype; f->msgbits = (uint8_t)msgbits;
            f->correctedbits = (uint8_t)corrected; f->fix_bit = (int8_t)fix_bit;
            f->flags = add_to_filter ? B200_FRAME_ICAO_ADDED : 0;
            memcpy(f->msg, msg, (size_t)msgbits / 8);
        } else overflow = 1;
        nfr++;
        j += (unsigned)msglen * 2; /* demod_2400.c:468; the loop adds the +1 */
    }

    st->samples_processed += mlen;
    st->buffers++;
    int flipped = 0;
    /* readsb.c:901,1227-1231: backgroundTasks() after each buffer, on the synthetic clock */
    if (o->ttl_ms > 0 && (!o->flip_armed || now_ms >= o->next_flip)) {
        oracle_icao_expire(o);
        o->next_flip = now_ms + o->ttl_ms; o->flip_armed = 1; flipped = 1;
    }
    if (res) {
        res->sample_timestamp = sample_ts; res->sum_level = sum_level; res->sum_power = sum_power;
        res->sum_signal_power = sum_sig; res->length = mlen; res->n_frames = nfr;
        res->buffer_seq = o->buffer_seq; res->icao_flipped = (uint32_t)flipped;
        res->demod_preambles = (uint32_t)(st->demod_preambles - before.demod_preambles);
        res->demod_rejected_bad = (uint32_t)(st->demod_rejected_bad - before.demod_rejected_bad);
        res->demod_rejected_unknown_icao = (uint32_t)(st->demod_rejected_unknown_icao - before.demod_rejected_unknown_icao);
        for (int i = 0; i < 2; i++) res->demod_accepted[i] = (uint32_t)(st->demod_accepted[i] - before.demod_accepted[i]);
        for (int i = 0; i < 5; i++) {
            res->demod_preamblePhase[i] = (uint32_t)(st->demod_preamblePhase[i] - before.demod_preamblePhase[i]);
            res->demod_bestPhase[i] = (uint32_t)(st->demod_bestPhase[i] - before.demod_bestPhase[i]);
        }
        res->pad_ = 0;
    }
    o->buffer_seq++;
    return overflow ? -1 : 0;
}

/* ------------------------------------------------------------------ demod_2400.c:575-761
 * Mode A/C: F1/F2 framing pulse pair 14 bit periods apart on a virtual 60 MHz clock (87 cycles per bit, 25 per sample),
 * 20 bit cells sliced against thresholds 3 dB either side of the geometric mean of noise and pulse level.
 * The float / double mix below is the reference's (float products, double for the +0.5 and the sqrt(2) factors). */
int oracle_demodulate2400AC(oracle_ctx *o, const uint16_t *m, unsigned mlen, int64_t sample_ts,
                            uint64_t sum_level, uint64_t sum_power, b200_modeac *out, unsigned cap, unsigned *n_out) {
    if (mlen == 0) return 0;
    const double mean_level = sum_level / 65536.0 / mlen;                 /* convert.c:100-102 */
    const double mean_power = sum_power / 65535.0 / 65535.0 / mlen;       /* convert.c:104-106 */
    return oracle_demodulate2400AC_levels(o, m, mlen, sample_ts, mean_level, mean_power, out, cap, n_out);
}

/* The same with mag_buf.mean_level / mean_power as the converter that filled the buffer returned them (any converter:
 * the sc16 ones return float-accumulated means, convert.c:243-249). */
int oracle_demodulate2400AC_levels(oracle_ctx *o, const uint16_t *m, unsigned mlen, int64_t sample_ts,
                                   double mean_level, double mean_power, b200_modeac *out, unsigned cap, unsigned *n_out) {
    int overflow = 0;
    if (mlen == 0) return 0;
    const double noise_stddev = sqrt(mean_power - mean_level * mean_level);   /* demod_2400.c:580 */
    const unsigned noise_level = (unsigned)((mean_power + noise_stddev) * 65535 + 0.5);
    for (unsigned f1 = 1; f1 < mlen; ++f1) {
        if (!(m[f1 - 1] < m[f1])) continue;                               /* rising edge */
        if (m[f1 + 2] > m[f1] || m[f1 + 2] > m[f1 + 1]) continue;         /* quiet part quiet enough */
        const unsigned f1_level = (m[f1] + m[f1 + 1]) / 2;
        if (noise_level * 2 > f1_level) continue;                         /* 6 dB above noise */
        const float f1a = (float)m[f1] * m[f1], f1b = (float)m[f1 + 1] * m[f1 + 1];
        const float fraction = f1b / (f1a + f1b);
        const unsigned f1_clock = (unsigned)(25 * (f1 + fraction * fraction) + 0.5);
        const unsigned f2_clock = f1_clock + 87 * 14, f2 = f2_clock / 25;
        if (!(m[f2 - 1] < m[f2])) continue;
        if (m[f2 + 2] > m[f2] || m[f2 + 2] > m[f2 + 1]) continue;
        const unsigned f2_level = (m[f2] + m[f2 + 1]) / 2;
        if (noise_level * 2 > f2_level) continue;
        const unsigned f1f2 = f1_level > f2_level ? f1_level : f2_level;
        const float midpoint = sqrtf(noise_level * f1f2);                 /* unsigned product, may wrap like the reference's */
        const unsigned signal_threshold = (unsigned)(midpoint * M_SQRT2 + 0.5);
        const unsigned noise_threshold = (unsigned)(midpoint / M_SQRT2 + 0.5);
        unsigned bits = 0, noisy = 0, uncertain = 0, clock = f1_clock;
        for (unsigned bit = 0; bit < 20; ++bit, clock += 87) {
            const unsigned s = clock / 25;
            bits <<= 1; noisy <<= 1; uncertain <<= 1;
            if (m[s + 2] >= signal_threshold) noisy |= 1;
            if (m[s] >= signal_threshold || m[s + 1] >= signal_threshold) bits |= 1;
            else if (m[s] > noise_threshold && m[s + 1] > noise_threshold) uncertain |= 1;
        }
        if ((bits & 0x80020) != 0x80020) continue;                        /* F1, F2 on */
        if ((bits & 0x0101B) != 0) continue;                              /* quiet cells off */
        if (noisy || uncertain) continue;
        const unsigned modeac =
            ((bits & 0x40000) ? 0x0010 : 0) | ((bits & 0x20000) ? 0x1000 : 0) | ((bits & 0x10000) ? 0x0020 : 0) |
            ((bits & 0x08000) ? 0x2000 : 0) | ((bits & 0x04000) ? 0x0040 : 0) | ((bits & 0x02000) ? 0x4000 : 0) |
            ((bits & 0x00800) ? 0x0100 : 0) | ((bits & 0x00400) ? 0x0001 : 0) | ((bits & 0x00200) ? 0x0200 : 0) |
            ((bits & 0x00100) ? 0x0002 : 0) | ((bits & 0x00080) ? 0x0400 : 0) | ((bits & 0x00040) ? 0x0004 : 0) |
            ((bits & 0x00004) ? 0x0080 : 0);
        if (*n_out < cap) {
            b200_modeac *a = &out[(*n_out)++];
            a->timestamp = sample_ts + f2_clock / 5; a->f1_sample = f1; a->modeac = (uint16_t)modeac; a->buffer_idx = 0;
        } else overflow = 1;
        f1 += 20 * 87 / 25;                                               /* skip the reply (the loop adds 1) */
        o->st.demod_modeac++;
    }
    return overflow ? -1 : 0;
}

/* ------------------------------------------------------------------ sdr_ifile.c:169-259 */
/* The receiver starts over (a frontend reopened): the next buffer's halo is zeros, like the first one of a stream. */
void oracle_stream_restart(oracle_ctx *o) { o->halo_valid = 0; }

long oracle_run_stream_uc8(oracle_ctx *o, const uint8_t *iq, uint64_t nsamples, unsigned buf_samples,
                           int64_t first_ts, b200_frame *frames, unsigned frame_cap,
                           b200_buffer_result *bufres, unsigned bufres_cap, unsigned *n_bufres) {
    uint16_t *data = malloc(((size_t)buf_samples + TRAIL) * 2);
    unsigned nf = 0, nb = 0;
    int bad = 0;
    for (uint64_t off = 0; off < nsamples; off += buf_samples) {
        unsigned len = (unsigned)((nsamples - off < buf_samples) ? nsamples - off : buf_samples);
        /* overlap copy, zeros when the previous buffer was too short (sdr_ifile.c:209-213) */
        if (o->halo_valid) memcpy(data, o->halo, TRAIL * 2); else memset(data, 0, TRAIL * 2);
        uint64_t sl, sp;
        oracle_convert_uc8(iq + off * 2, data + TRAIL, len, &sl, &sp);
        b200_buffer_result r;
        if (oracle_demodulate2400(o, data, len, first_ts + (int64_t)off * 5, sl, sp, frames, frame_cap, &nf, &r) < 0) bad = 1;
        if (nb < bufres_cap && bufres) bufres[nb] = r;
        nb++;
        if (len >= TRAIL) { memcpy(o->halo, data + len, TRAIL * 2); o->halo_valid = 1; } else o->halo_valid = 0;
    }
    free(data);
    if (n_bufres) *n_bufres = nb;
    return bad ? -1 : (long)nf;
}

/* ------------------------------------------------------------------ net_io.c:1617-1648, 1655-1714
 * Beast binary record of one accepted frame, as modesSendBeastOutput writes it for a net_writer without receiverId:
 * 0x1a, type ('2' 56-bit, '3' 112-bit, '1' Mode A/C), 6-byte big-endian 12 MHz timestamp, one signal byte, the frame;
 * every 0x1a after the type byte is doubled.  verbatim = Modes.net_verbatim: the bytes as received (mm->verbatim) instead
 * of the corrected frame. */
static uint8_t *beast_put(uint8_t *p, uint8_t ch) { *p++ = ch; if (ch == 0x1a) *p++ = ch; return p; }

static uint8_t *beast_head(uint8_t *p, char type, int64_t timestamp, double signal_level) {
    *p++ = 0x1a; *p++ = (uint8_t)type;
    for (int sh = 40; sh >= 0; sh -= 8) p = beast_put(p, (uint8_t)(timestamp >> sh));
    int sig = (int)nearbyint(sqrt(signal_level) * 255);
    if (signal_level > 0 && sig < 1) sig = 1;
    if (sig > 255) sig = 255;
    return beast_put(p, (uint8_t)sig);
}

unsigned oracle_beast_frame(const b200_frame *f, int verbatim, uint8_t *out) {
    uint8_t msg[14];
    memcpy(msg, f->msg, 14);
    if (verbatim && f->fix_bit >= 0) msg[f->fix_bit >> 3] ^= (uint8_t)(1u << (7 - (f->fix_bit & 7)));
    const int len = f->msgbits / 8;
    /* demod_2400.c:448-457: signalLevel = sum / 65535 / 65535 / signal_len */
    const double signal_level = (double)f->sigpow_sum / 65535.0 / 65535.0 / f->signal_len;
    uint8_t *p = beast_head(out, len == 7 ? '2' : '3', f->timestamp, signal_level);
    for (int i = 0; i < len; i++) p = beast_put(p, msg[i]);
    return (unsigned)(p - out);
}

unsigned oracle_beast_modeac(const b200_modeac *a, uint8_t *out) {
    /* mode_ac.c:171-173: two bytes, Mode A word big-endian; signalLevel is never set for Mode A/C (netGetMM zeroes it) */
    uint8_t *p = beast_head(out, '1', a->timestamp, 0.0);
    p = beast_put(p, (uint8_t)(a->modeac >> 8));
    p = beast_put(p, (uint8_t)a->modeac);
    return (unsigned)(p - out);
}

/* ------------------------------------------------------------------ convert.c:212-250 (sc16) and 329-367 (sc16q11)
 * The float-path converters.  Magnitude per sample exactly as the reference computes it; the two float accumulators are
 * added to in sample order (sum_power first, then sum_level) and handed back as floats:
 * mean_level = sum_level / nsamples, mean_power = sum_power / nsamples (float divisions, then widened to double). */
void oracle_convert_sc16(const int16_t *iq, uint16_t *mag_out, unsigned nsamples, int q11, float *sum_level_out, float *sum_power_out) {
    const float scale = q11 ? 2048.0f : 32768.0f;
    float sum_level = 0, sum_power = 0;
    for (unsigned i = 0; i < nsamples; i++) {
        const int16_t I = iq[2 * i], Q = iq[2 * i + 1];
        const float fI = I / scale, fQ = Q / scale;
        float magsq = fI * fI + fQ * fQ;
        if (magsq > 1) magsq = 1;
        const float mag = sqrtf(magsq);
        sum_power += magsq;
        sum_level += mag;
        mag_out[i] = (uint16_t)(mag * 65535.0f + 0.5f);
    }
    *sum_level_out = sum_level; *sum_power_out = sum_power;
}
