/*
 * idn_oracle.c -- CPU restatement of idencomp's rANS hot path.  TEST INFRASTRUCTURE ONLY
 * (see idn_oracle.h for the rules and the parity status).  Plain C11 + zlib + pthreads.
 *
 * Reference paths are relative to /root/reference/idencomp/src unless stated.
 */
#define _GNU_SOURCE
#include "idn_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>

static _Thread_local char g_err[256];
const char *orc_last_error(void) { return g_err; }
static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

uint32_t orc_crc32(uint32_t crc, const uint8_t *p, size_t n) {
    /* crc32fast 1.3.2 == CRC-32/IEEE == zlib crc32 (SURVEY.md 8c) */
    while (n > 0) {
        uInt chunk = n > 0x40000000u ? 0x40000000u : (uInt)n;
        crc = (uint32_t)crc32(crc, p, chunk);
        p += chunk;
        n -= chunk;
    }
    return crc;
}

/* ------------------------------------------------------------------------------------------------
 * a1  Context::as_integer_cum_freqs + fix_zero_freqs      context.rs:346-394
 * ---------------------------------------------------------------------------------------------- */
void orc_quantise(const float *probs, int nsym, int scale_bits, uint32_t *cum_out) {
    uint32_t total = 1u << scale_bits;
    volatile float acc = 0.0f; /* volatile: keep every step rounded to f32 (no x87/FMA contraction) */
    uint32_t freq[256];
    for (int i = 0; i < nsym; i++) {
        float raw = acc; /* scan yields the accumulator BEFORE adding x (context.rs:356-360) */
        volatile float scaled = probs[i] * (float)total;
        acc = acc + scaled;
        cum_out[i] = (uint32_t)roundf(raw); /* Rust f32::round = half away from zero = C roundf */
    }
    /* cum_freq_to_freq (context.rs:411-417) */
    for (int i = 0; i < nsym - 1; i++) freq[i] = cum_out[i + 1] - cum_out[i];
    freq[nsym - 1] = total - cum_out[nsym - 1];
    /* fix_zero_freqs (context.rs:373-394) */
    int zero_count = 0;
    for (int i = 0; i < nsym; i++)
        if (freq[i] == 0) {
            freq[i] = 1;
            zero_count++;
        }
    int i = 0;
    while (zero_count > 0) {
        if (freq[i] > 1) {
            freq[i]--;
            zero_count--;
        }
        i++;
        if (i >= nsym) i = 0;
    }
    /* freq_to_cum_freq (context.rs:433-440) */
    uint32_t a = 0;
    for (int k = 0; k < nsym; k++) {
        cum_out[k] = a;
        a += freq[k];
    }
}

/* ------------------------------------------------------------------------------------------------
 * a4/a5  context-spec generators     context_spec.rs:218-529, int_queue.rs:1-86
 * ---------------------------------------------------------------------------------------------- */
static uint32_t ipow(uint32_t b, uint32_t e) {
    uint32_t r = 1;
    while (e--) r *= b;
    return r;
}
static uint32_t bitlen(uint32_t v) {
    uint32_t n = 0;
    while (v) {
        n++;
        v >>= 1;
    }
    return n;
}
/* IntQueue::num_bits  int_queue.rs:40-43: 32 - leading_zeros(B^n - 1) */
static uint32_t queue_bits(uint32_t base, uint32_t n) { return bitlen(ipow(base, n) - 1u); }

/* serde names: idencomp-macros/src/lib.rs:166-196 */
int orc_spec_parse(const char *name, orc_spec_t *out) {
    int ao, qo, pb, qm;
    char tail;
    memset(out, 0, sizeof *out);
    if (strcmp(name, "dummy") == 0) {
        out->kind = ORC_KIND_GENERIC;
        return 0;
    }
    if (sscanf(name, "generic_ao%d_qo%d_pb%d%c", &ao, &qo, &pb, &tail) == 3) {
        out->kind = ORC_KIND_GENERIC;
        out->ao = ao;
        out->qo = qo;
        out->pb = pb;
        return 0;
    }
    if (sscanf(name, "light_ao%d_qo%d_pb%d_qm%d%c", &ao, &qo, &pb, &qm, &tail) == 4) {
        out->kind = ORC_KIND_LIGHT;
        out->ao = ao;
        out->qo = qo;
        out->pb = pb;
        out->qmax = qm;
        return 0;
    }
    return -1;
}

static void spec_bases(const orc_spec_t *s, uint32_t *ba, uint32_t *bq) {
    if (s->kind == ORC_KIND_LIGHT) {
        *ba = 4; /* context_spec.rs:428 IntQueue<4, ACID_ORDER> */
        *bq = (uint32_t)s->qmax;
    } else {
        *ba = 5; /* context_spec.rs:225-226 */
        *bq = 94;
    }
}

uint32_t orc_spec_bits(const orc_spec_t *s) {
    uint32_t ba, bq;
    spec_bases(s, &ba, &bq);
    return queue_bits(ba, (uint32_t)s->ao) + queue_bits(bq, (uint32_t)s->qo) + (uint32_t)s->pb;
}
uint64_t orc_spec_num(const orc_spec_t *s) { return 1ull << orc_spec_bits(s); }

void orc_gen_init(orc_gen_t *g, const orc_spec_t *s, uint32_t length) {
    memset(g, 0, sizeof *g);
    g->spec = *s;
    spec_bases(s, &g->base_a, &g->base_q);
    g->abits = queue_bits(g->base_a, (uint32_t)s->ao);
    g->qbits = queue_bits(g->base_q, (uint32_t)s->qo);
    g->last_pow_a = s->ao ? ipow(g->base_a, (uint32_t)s->ao - 1) : 0;
    g->last_pow_q = s->qo ? ipow(g->base_q, (uint32_t)s->qo - 1) : 0;
    g->length = length;
    /* initial queue state is 0 whatever the default symbol: calc_default_state returns 0 at depth 0
     * (int_queue.rs:24-30) */
}

/* current_context: context_spec.rs:377-383 (generic), 508-514 (light); position(): 313-316 */
uint32_t orc_gen_current(const orc_gen_t *g) {
    uint32_t pos = (uint32_t)(g->position * (1u << g->spec.pb)) / g->length; /* u32 arithmetic */
    uint32_t v = g->qstate;
    v = (v << g->abits) | g->astate;
    v = (v << g->spec.pb) | pos;
    return v;
}

/* update: context_spec.rs:385-389 (generic), 516-529 (light); with_pushed_back int_queue.rs:63-70 */
void orc_gen_update(orc_gen_t *g, uint8_t acid, uint8_t q) {
    uint32_t va = acid, vq = q;
    if (g->spec.kind == ORC_KIND_LIGHT) {
        if (acid == 0 || q == 0) {
            va = 0;
            vq = 0;
        } else {
            va = (uint32_t)acid - 1;
            vq = (uint32_t)q * (uint32_t)g->spec.qmax / 94u;
        }
    }
    if (g->spec.ao) g->astate = g->astate % g->last_pow_a * g->base_a + va;
    if (g->spec.qo) g->qstate = g->qstate % g->last_pow_q * g->base_q + vq;
    g->position += 1;
}

/* ------------------------------------------------------------------------------------------------
 * ryg rans_byte.h restated (crate rans 0.2.1 / ryg-rans-sys 1.0.7; call sites compressor.rs:1-193)
 * ---------------------------------------------------------------------------------------------- */
#define RANS_L (1u << 23)

typedef struct {
    uint32_t x_max, rcp_freq, bias;
    uint16_t cmpl_freq, rcp_shift;
} enc_sym_t;

static void enc_sym_init(enc_sym_t *s, uint32_t start, uint32_t freq, uint32_t scale_bits) {
    s->x_max = ((RANS_L >> scale_bits) << 8) * freq;
    s->cmpl_freq = (uint16_t)((1u << scale_bits) - freq);
    if (freq < 2) {
        s->rcp_freq = ~0u;
        s->rcp_shift = 0;
        s->bias = start + (1u << scale_bits) - 1;
    } else {
        uint32_t shift = 0;
        while (freq > (1u << shift)) shift++;
        s->rcp_freq = (uint32_t)(((1ull << (shift + 31)) + freq - 1) / freq);
        s->rcp_shift = (uint16_t)(shift - 1);
        s->bias = start;
    }
}

static inline void enc_put(uint32_t *r, uint8_t **pptr, const enc_sym_t *sym) {
    uint32_t x = *r;
    uint32_t x_max = sym->x_max;
    if (x >= x_max) {
        uint8_t *ptr = *pptr;
        do {
            *--ptr = (uint8_t)(x & 0xff);
            x >>= 8;
        } while (x >= x_max);
        *pptr = ptr;
    }
    uint32_t q = (uint32_t)(((uint64_t)x * sym->rcp_freq) >> 32) >> sym->rcp_shift;
    *r = x + sym->bias + q * sym->cmpl_freq;
}

static inline void enc_flush(uint32_t x, uint8_t **pptr) {
    uint8_t *ptr = *pptr - 4;
    ptr[0] = (uint8_t)(x >> 0);
    ptr[1] = (uint8_t)(x >> 8);
    ptr[2] = (uint8_t)(x >> 16);
    ptr[3] = (uint8_t)(x >> 24);
    *pptr = ptr;
}

size_t orc_rans_encode_raw(const uint32_t *starts, const uint32_t *freqs, size_t n, int nstates,
                           int scale_bits, uint8_t *out) {
    size_t cap = 2 * n + 4 * (size_t)nstates;
    uint8_t *tmp = (uint8_t *)malloc(cap);
    uint8_t *ptr = tmp + cap;
    uint32_t st[8];
    for (int i = 0; i < nstates; i++) st[i] = RANS_L;
    for (size_t i = 0; i < n; i++) {
        enc_sym_t s;
        enc_sym_init(&s, starts[i], freqs[i], (uint32_t)scale_bits);
        enc_put(&st[i % (size_t)nstates], &ptr, &s);
    }
    for (int i = 0; i < nstates; i++) enc_flush(st[i], &ptr);
    size_t len = (size_t)(tmp + cap - ptr);
    memcpy(out, ptr, len);
    free(tmp);
    return len;
}

/* ------------------------------------------------------------------------------------------------
 * a2/a3  model tables
 * ---------------------------------------------------------------------------------------------- */
struct orc_model {
    int type;
    uint32_t nsym, n_ctx; /* n_ctx excludes the dummy row 0 */
    orc_spec_t spec;
    uint8_t id[32];
    uint16_t *cum;  /* [(n_ctx+1)][nsym+1], row 0 = Context::dummy (sequence_compressor.rs:26-29) */
    enc_sym_t *enc; /* [(n_ctx+1)][nsym]  RansEncContext (compressor.rs:21-35) */
    uint8_t *lut;   /* optional slot->symbol [(n_ctx+1)][1<<14]  (compressor.rs:124-128) */
    /* map: dense when spec_num <= 2^24, else open-addressing hash (sequence_compressor.rs:37-40) */
    uint64_t spec_num;
    uint32_t *dense;
    uint32_t *hkeys, *hvals;
    uint32_t hmask;
};

static uint32_t hash32(uint32_t k) {
    k ^= k >> 16;
    k *= 0x7feb352dU;
    k ^= k >> 15;
    k *= 0x846ca68bU;
    k ^= k >> 16;
    return k;
}

orc_model_t *orc_model_new(int type, const char *spec_name, uint32_t n_ctx, const float *probs,
                           const uint32_t *spec_keys, const uint32_t *spec_ctx, size_t n_specs,
                           const uint8_t identifier[32]) {
    orc_model_t *m = (orc_model_t *)calloc(1, sizeof *m);
    if (!m) return NULL;
    m->type = type;
    m->nsym = type == ORC_TYPE_ACID ? ORC_ACID_SYMS : ORC_Q_SYMS;
    m->n_ctx = n_ctx;
    if (identifier) memcpy(m->id, identifier, 32);
    if (orc_spec_parse(spec_name, &m->spec) != 0 || n_ctx > 65536 /* check_model :209-219 */) {
        free(m);
        return NULL;
    }
    uint32_t ns = m->nsym;
    size_t rows = (size_t)n_ctx + 1;
    m->cum = (uint16_t *)malloc(rows * (ns + 1) * sizeof(uint16_t));
    m->enc = (enc_sym_t *)malloc(rows * ns * sizeof(enc_sym_t));
    float dummy[ORC_Q_SYMS];
    for (uint32_t i = 0; i < ns; i++) dummy[i] = 1.0f / (float)ns; /* context.rs:225-229 */
    uint32_t cum[ORC_Q_SYMS + 1];
    for (size_t r = 0; r < rows; r++) {
        orc_quantise(r == 0 ? dummy : probs + (r - 1) * ns, (int)ns, ORC_SCALE_BITS, cum);
        cum[ns] = 1u << ORC_SCALE_BITS;
        for (uint32_t s = 0; s <= ns; s++) m->cum[r * (ns + 1) + s] = (uint16_t)cum[s];
        for (uint32_t s = 0; s < ns; s++)
            enc_sym_init(&m->enc[r * ns + s], cum[s], cum[s + 1] - cum[s], ORC_SCALE_BITS);
    }
    if (ns == ORC_Q_SYMS && rows <= 4096) {
        m->lut = (uint8_t *)malloc(rows << ORC_SCALE_BITS);
        for (size_t r = 0; r < rows; r++) {
            const uint16_t *c = m->cum + r * (ns + 1);
            uint8_t *l = m->lut + (r << ORC_SCALE_BITS);
            for (uint32_t s = 0; s < ns; s++)
                for (uint32_t k = c[s]; k < c[s + 1]; k++) l[k] = (uint8_t)s;
        }
    }
    m->spec_num = orc_spec_num(&m->spec);
    if (m->spec_num <= (1ull << 24)) {
        m->dense = (uint32_t *)calloc((size_t)m->spec_num, sizeof(uint32_t));
        for (size_t i = 0; i < n_specs; i++)
            if (spec_keys[i] < m->spec_num) m->dense[spec_keys[i]] = spec_ctx[i] + 1;
    } else {
        uint32_t cap = 16;
        while (cap < n_specs * 2 + 1) cap <<= 1;
        m->hmask = cap - 1;
        m->hkeys = (uint32_t *)malloc(cap * sizeof(uint32_t));
        m->hvals = (uint32_t *)calloc(cap, sizeof(uint32_t)); /* 0 = empty slot */
        for (size_t i = 0; i < n_specs; i++) {
            uint32_t h = hash32(spec_keys[i]) & m->hmask;
            while (m->hvals[h] != 0 && m->hkeys[h] != spec_keys[i]) h = (h + 1) & m->hmask;
            m->hkeys[h] = spec_keys[i];
            m->hvals[h] = spec_ctx[i] + 1;
        }
    }
    return m;
}

void orc_model_free(orc_model_t *m) {
    if (!m) return;
    free(m->cum);
    free(m->enc);
    free(m->lut);
    free(m->dense);
    free(m->hkeys);
    free(m->hvals);
    free(m);
}
int orc_model_type(const orc_model_t *m) { return m->type; }
uint32_t orc_model_nctx(const orc_model_t *m) { return m->n_ctx; }
uint32_t orc_model_nsym(const orc_model_t *m) { return m->nsym; }
void orc_model_identifier(const orc_model_t *m, uint8_t out[32]) { memcpy(out, m->id, 32); }
void orc_model_cum_row(const orc_model_t *m, uint32_t ctx, uint32_t *out) {
    for (uint32_t s = 0; s <= m->nsym; s++) out[s] = m->cum[(size_t)ctx * (m->nsym + 1) + s];
}

/* context_for: sequence_compressor.rs:60-62, 203-205 */
static inline uint32_t ctx_for(const orc_model_t *m, uint32_t spec) {
    if (m->dense) return m->dense[spec];
    uint32_t h = hash32(spec) & m->hmask;
    while (m->hvals[h] != 0) {
        if (m->hkeys[h] == spec) return m->hvals[h];
        h = (h + 1) & m->hmask;
    }
    return 0;
}
uint32_t orc_model_ctx_for(const orc_model_t *m, uint32_t spec) { return ctx_for(m, spec); }

/* ------------------------------------------------------------------------------------------------
 * a8  SequenceCompressor::compress   sequence_compressor.rs:82-155 ; RansCompressor<2> compressor.rs:83-98
 * ---------------------------------------------------------------------------------------------- */
size_t orc_encode_read(const orc_model_t *am, const orc_model_t *qm, const uint8_t *acids,
                       const uint8_t *quals, uint32_t len, uint8_t *out) {
    size_t cap = 4 * (size_t)len + 8;
    uint32_t *ctx_a = (uint32_t *)malloc(((size_t)len + 1) * 2 * sizeof(uint32_t));
    uint32_t *ctx_q = ctx_a + len + 1;
    uint8_t *tmp = (uint8_t *)malloc(cap);
    /* gen_contexts (:126-155): both generators are fed the TRUE (acid, q) pair, forward */
    orc_gen_t ga, gq;
    orc_gen_init(&ga, &am->spec, len);
    orc_gen_init(&gq, &qm->spec, len);
    for (uint32_t i = 0; i < len; i++) {
        ctx_a[i] = ctx_for(am, orc_gen_current(&ga));
        ctx_q[i] = ctx_for(qm, orc_gen_current(&gq));
        orc_gen_update(&ga, acids[i], quals[i]);
        orc_gen_update(&gq, acids[i], quals[i]);
    }
    /* reverse put (:92-121): put_at(0, acid) then put_at(1, q) (compressor.rs:95-96) */
    uint32_t s0 = RANS_L, s1 = RANS_L;
    uint8_t *ptr = tmp + cap;
    for (uint32_t i = len; i-- > 0;) {
        enc_put(&s0, &ptr, &am->enc[(size_t)ctx_a[i] * ORC_ACID_SYMS + acids[i]]);
        enc_put(&s1, &ptr, &qm->enc[(size_t)ctx_q[i] * ORC_Q_SYMS + quals[i]]);
    }
    /* flush_all: state 0 first, then state 1; the buffer grows downward */
    enc_flush(s0, &ptr);
    enc_flush(s1, &ptr);
    size_t n = (size_t)(tmp + cap - ptr);
    memcpy(out, ptr, n);
    free(tmp);
    free(ctx_a);
    return n;
}

/* slot -> symbol (cum_freq_to_symbol_index compressor.rs:137-139) */
static inline uint32_t find_sym(const orc_model_t *m, uint32_t ctx, uint32_t slot) {
    if (m->lut) return m->lut[((size_t)ctx << ORC_SCALE_BITS) + slot];
    const uint16_t *c = m->cum + (size_t)ctx * (m->nsym + 1);
    uint32_t lo = 0, hi = m->nsym; /* largest s with c[s] <= slot */
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (c[mid] <= slot)
            lo = mid;
        else
            hi = mid;
    }
    return lo;
}

/* a9  SequenceDecompressor::decompress  sequence_compressor.rs:231-278 ; RansDecompressor<2>::get
 * compressor.rs:173-193.  Out-of-bounds reads are refused (the reference trusts the lengths). */
int orc_decode_read(const orc_model_t *am, const orc_model_t *qm, const uint8_t *data, size_t n,
                    uint32_t len, uint8_t *acids, uint8_t *quals, uint32_t final_states[2],
                    size_t *consumed) {
    if (n < 8) return fail(ORC_E_SERIALIZE, "sequence payload shorter than 8 bytes");
    const uint32_t mask = (1u << ORC_SCALE_BITS) - 1;
    /* decoder state 0 <- bytes[0..4] (q-scores), state 1 <- bytes[4..8] (acids) */
    uint32_t sq = (uint32_t)data[0] | (uint32_t)data[1] << 8 | (uint32_t)data[2] << 16 | (uint32_t)data[3] << 24;
    uint32_t sa = (uint32_t)data[4] | (uint32_t)data[5] << 8 | (uint32_t)data[6] << 16 | (uint32_t)data[7] << 24;
    size_t p = 8;
    orc_gen_t ga, gq;
    orc_gen_init(&ga, &am->spec, len);
    orc_gen_init(&gq, &qm->spec, len);
    for (uint32_t i = 0; i < len; i++) {
        uint32_t ca = ctx_for(am, orc_gen_current(&ga));
        uint32_t cq = ctx_for(qm, orc_gen_current(&gq));
        uint32_t slot_q = sq & mask, slot_a = sa & mask;
        uint32_t yq = find_sym(qm, cq, slot_q);
        uint32_t ya = find_sym(am, ca, slot_a);
        const uint16_t *rq = qm->cum + (size_t)cq * (ORC_Q_SYMS + 1);
        const uint16_t *ra = am->cum + (size_t)ca * (ORC_ACID_SYMS + 1);
        sq = (uint32_t)(rq[yq + 1] - rq[yq]) * (sq >> ORC_SCALE_BITS) + slot_q - rq[yq];
        sa = (uint32_t)(ra[ya + 1] - ra[ya]) * (sa >> ORC_SCALE_BITS) + slot_a - ra[ya];
        while (sq < RANS_L) { /* renorm_all: state 0 (q) first, then state 1 (acid) */
            if (p >= n) return fail(ORC_E_SERIALIZE, "sequence payload exhausted");
            sq = (sq << 8) | data[p++];
        }
        while (sa < RANS_L) {
            if (p >= n) return fail(ORC_E_SERIALIZE, "sequence payload exhausted");
            sa = (sa << 8) | data[p++];
        }
        acids[i] = (uint8_t)ya;
        quals[i] = (uint8_t)yq;
        orc_gen_update(&ga, (uint8_t)ya, (uint8_t)yq);
        orc_gen_update(&gq, (uint8_t)ya, (uint8_t)yq);
    }
    if (final_states) {
        final_states[0] = sq;
        final_states[1] = sa;
    }
    if (consumed) *consumed = p;
    return ORC_OK;
}

/* a6  ModelTester::compute_size   idn/model_chooser.rs:215-243: forward order, one state */
size_t orc_score_read(const orc_model_t *m, const uint8_t *acids, const uint8_t *quals, uint32_t len) {
    orc_gen_t g;
    orc_gen_init(&g, &m->spec, len);
    uint32_t x = RANS_L;
    size_t bytes = 0;
    const uint8_t *syms = m->type == ORC_TYPE_ACID ? acids : quals;
    for (uint32_t i = 0; i < len; i++) {
        const enc_sym_t *s = &m->enc[(size_t)ctx_for(m, orc_gen_current(&g)) * m->nsym + syms[i]];
        while (x >= s->x_max) {
            x >>= 8;
            bytes++;
        }
        uint32_t q = (uint32_t)(((uint64_t)x * s->rcp_freq) >> 32) >> s->rcp_shift;
        x = x + s->bias + q * s->cmpl_freq;
        orc_gen_update(&g, acids[i], quals[i]);
    }
    return bytes + 4;
}

/* ------------------------------------------------------------------------------------------------
 * buffers
 * ---------------------------------------------------------------------------------------------- */
static int buf_reserve(orc_buf_t *b, size_t extra) {
    if (b->len + extra <= b->cap) return 0;
    size_t nc = b->cap ? b->cap : 4096;
    while (nc < b->len + extra) nc *= 2;
    uint8_t *nd = (uint8_t *)realloc(b->data, nc);
    if (!nd) return -1;
    b->data = nd;
    b->cap = nc;
    return 0;
}
static void buf_put(orc_buf_t *b, const void *p, size_t n) {
    buf_reserve(b, n);
    memcpy(b->data + b->len, p, n);
    b->len += n;
}
static void buf_u8(orc_buf_t *b, uint8_t v) { buf_put(b, &v, 1); }
static void buf_u32be(orc_buf_t *b, uint32_t v) {
    uint8_t t[4] = {(uint8_t)(v >> 24), (uint8_t)(v >> 16), (uint8_t)(v >> 8), (uint8_t)v};
    buf_put(b, t, 4);
}
void orc_buf_free(orc_buf_t *b) {
    free(b->data);
    b->data = NULL;
    b->len = b->cap = 0;
}

/* ------------------------------------------------------------------------------------------------
 * a7  greedy per-read model choice   idn/model_chooser.rs:168-198, idn/compressor_block.rs:232-280
 * returns the provider index of the chosen model of `type`; *bytes = size + penalty of the winner
 * ---------------------------------------------------------------------------------------------- */
static int choose_model(const orc_params_t *p, int type, int current, const uint8_t *acids,
                        const uint8_t *quals, uint32_t len, size_t *bytes) {
    int best = -1;
    size_t best_len = 0;
    for (uint32_t k = 0; k < p->n_models; k++) {
        if (p->models[k]->type != type) continue;
        size_t l = orc_score_read(p->models[k], acids, quals, len);
        /* penalty compares model IDENTIFIERS (model_chooser.rs:181); identifiers are unique per index */
        if ((int)k != current) l += 2;
        if (best < 0 || l < best_len) { /* Iterator::min_by keeps the FIRST minimum */
            best = (int)k;
            best_len = l;
        }
    }
    *bytes = best_len;
    return best;
}

/* names slice: compressor_block.rs:146-206 (Deflate branch; flate2 default level 6, raw deflate) */
static int deflate_names(const uint8_t *src, size_t n, int level, orc_buf_t *out) {
    z_stream z;
    memset(&z, 0, sizeof z);
    if (deflateInit2(&z, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK)
        return fail(ORC_E_IO, "deflateInit2 failed");
    uLong bound = deflateBound(&z, (uLong)n) + 64;
    buf_reserve(out, bound);
    z.next_in = (Bytef *)src;
    z.avail_in = (uInt)n;
    z.next_out = out->data + out->len;
    z.avail_out = (uInt)bound;
    int rc = deflate(&z, Z_FINISH);
    deflateEnd(&z);
    if (rc != Z_STREAM_END) return fail(ORC_E_IO, "deflate failed (%d)", rc);
    out->len += bound - z.avail_out;
    return ORC_OK;
}

static int inflate_names(const uint8_t *src, size_t n, orc_buf_t *out) {
    z_stream z;
    memset(&z, 0, sizeof z);
    if (inflateInit2(&z, -15) != Z_OK) return fail(ORC_E_IO, "inflateInit2 failed");
    z.next_in = (Bytef *)src;
    z.avail_in = (uInt)n;
    int rc;
    do {
        buf_reserve(out, 65536);
        z.next_out = out->data + out->len;
        z.avail_out = (uInt)(out->cap - out->len);
        size_t before = z.avail_out;
        rc = inflate(&z, Z_NO_FLUSH);
        out->len += before - z.avail_out;
    } while (rc == Z_OK);
    inflateEnd(&z);
    if (rc != Z_STREAM_END) return fail(ORC_E_IO, "inflate failed (%d)", rc);
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------------
 * a10  IdnBlockCompressor::prepare_to_write   idn/compressor_block.rs:83-120 ; BlockWriter writer_block.rs
 * ---------------------------------------------------------------------------------------------- */
int orc_compress_block(const orc_params_t *p, const orc_reads_t *in, uint64_t first_read,
                       uint64_t n_reads, orc_buf_t *out, uint32_t *crc_out, orc_stats_t *stats) {
    uint32_t crc = 0;
    *crc_out = 0;
    if (n_reads == 0) return ORC_OK; /* :84-86 */
    if (p->include_identifiers) {
        if (p->quality >= 8) return fail(ORC_E_UNSUPPORTED, "Brotli name slices are not restated");
        const uint8_t *nb = in->names;
        uint64_t a = in->name_off ? in->name_off[first_read] : 0;
        orc_buf_t joined = {0};
        for (uint64_t r = first_read; r < first_read + n_reads; r++) {
            if (r > first_read) buf_u8(&joined, '\n'); /* identifiers_as_lines :199-206 */
            if (in->name_off) buf_put(&joined, nb + in->name_off[r], in->name_off[r + 1] - in->name_off[r]);
        }
        (void)a;
        orc_buf_t z = {0};
        int rc = deflate_names(joined.data, joined.len, p->deflate_level ? p->deflate_level : 6, &z);
        if (rc) {
            orc_buf_free(&joined);
            orc_buf_free(&z);
            return rc;
        }
        buf_u8(out, 0x00); /* IdnSliceHeader::Identifiers  data.rs:46-47 */
        buf_u32be(out, (uint32_t)z.len);
        buf_u8(out, 1); /* IdnIdentifierCompression::Deflate  data.rs:57-61 */
        buf_put(out, z.data, z.len);
        if (stats) stats->names_bytes += z.len;
        orc_buf_free(&joined);
        orc_buf_free(&z);
    }
    int cur_a = -1, cur_q = -1;
    int def_a = -1, def_q = -1;
    for (uint32_t k = 0; k < p->n_models; k++) {
        if (p->models[k]->type == ORC_TYPE_ACID && def_a < 0) def_a = (int)k;
        if (p->models[k]->type == ORC_TYPE_QSCORE && def_q < 0) def_q = (int)k;
    }
    if (def_a < 0 || def_q < 0) return fail(ORC_E_INVALID_STATE, "need at least one model per type");
    if (p->fast) {
        if (p->n_models != 2) return fail(ORC_E_INVALID_STATE, "fast mode needs exactly 2 models"); /* :96 */
        buf_u8(out, 0x01);
        buf_u8(out, 0);
        buf_u8(out, 0x01);
        buf_u8(out, 1);
    }
    uint8_t *payload = NULL;
    size_t payload_cap = 0;
    for (uint64_t r = first_read; r < first_read + n_reads; r++) {
        const uint8_t *ac = in->acids + in->read_off[r];
        const uint8_t *qu = in->quals + in->read_off[r];
        uint32_t len = (uint32_t)(in->read_off[r + 1] - in->read_off[r]);
        int ma = def_a, mq = def_q;
        if (!p->fast) {
            size_t bytes;
            ma = choose_model(p, ORC_TYPE_ACID, cur_a, ac, qu, len, &bytes); /* acid first :103-104 */
            if (ma != cur_a) {
                buf_u8(out, 0x01); /* SwitchModel  data.rs:48-49 */
                buf_u8(out, (uint8_t)ma);
                cur_a = ma;
                if (stats) stats->acid_switches++;
            }
            if (stats) stats->out_acid_bytes += bytes;
            mq = choose_model(p, ORC_TYPE_QSCORE, cur_q, ac, qu, len, &bytes);
            if (mq != cur_q) {
                buf_u8(out, 0x01);
                buf_u8(out, (uint8_t)mq);
                cur_q = mq;
                if (stats) stats->q_switches++;
            }
            if (stats) stats->out_q_score_bytes += bytes;
        }
        if (payload_cap < 4 * (size_t)len + 8) {
            payload_cap = 4 * (size_t)len + 8;
            payload = (uint8_t *)realloc(payload, payload_cap);
        }
        size_t n = orc_encode_read(p->models[ma], p->models[mq], ac, qu, len, payload);
        /* sequence.hash -> crc: name bytes, acid bytes, q bytes   sequence.rs:381-394, writer_block.rs:64 */
        if (in->name_off && p->include_identifiers)
            crc = orc_crc32(crc, in->names + in->name_off[r], in->name_off[r + 1] - in->name_off[r]);
        crc = orc_crc32(crc, ac, len);
        crc = orc_crc32(crc, qu, len);
        buf_u8(out, 0x02); /* Sequence slice  data.rs:50-51, 79-84 */
        buf_u32be(out, (uint32_t)n);
        buf_u32be(out, len);
        buf_put(out, payload, n);
    }
    free(payload);
    *crc_out = crc;
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------------
 * block worker pool (stands in for idn/thread_pool.rs + IdnBlockLock ordered commit common.rs:10-57)
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int (*fn)(void *ctx, uint64_t i);
    void *ctx;
    uint64_t n;
    uint64_t next;
    int err;
    char errmsg[256];
    pthread_mutex_t mu;
} pool_job_t;

static void *pool_worker(void *arg) {
    pool_job_t *j = (pool_job_t *)arg;
    for (;;) {
        pthread_mutex_lock(&j->mu);
        uint64_t i = j->next++;
        int stop = j->err != 0;
        pthread_mutex_unlock(&j->mu);
        if (i >= j->n || stop) break;
        int rc = j->fn(j->ctx, i);
        if (rc) {
            pthread_mutex_lock(&j->mu);
            if (!j->err) {
                j->err = rc;
                snprintf(j->errmsg, sizeof j->errmsg, "%s", g_err);
            }
            pthread_mutex_unlock(&j->mu);
        }
    }
    return NULL;
}

static int pool_run(int threads, uint64_t n, int (*fn)(void *, uint64_t), void *ctx) {
    pool_job_t j;
    memset(&j, 0, sizeof j);
    j.fn = fn;
    j.ctx = ctx;
    j.n = n;
    pthread_mutex_init(&j.mu, NULL);
    if (threads <= 1 || n <= 1) {
        pool_worker(&j);
    } else {
        if ((uint64_t)threads > n) threads = (int)n;
        pthread_t *t = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
        for (int i = 0; i < threads; i++) pthread_create(&t[i], NULL, pool_worker, &j);
        for (int i = 0; i < threads; i++) pthread_join(t[i], NULL);
        free(t);
    }
    pthread_mutex_destroy(&j.mu);
    if (j.err) snprintf(g_err, sizeof g_err, "%s", j.errmsg);
    return j.err;
}

/* ------------------------------------------------------------------------------------------------
 * whole-file compress
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    const orc_params_t *p;
    const orc_reads_t *in;
    const uint64_t *blk_first; /* [n_blocks+1] */
    orc_buf_t *blk_out;
    uint32_t *blk_crc;
    orc_stats_t *blk_stats;
} cjob_t;

static int compress_one(void *vctx, uint64_t b) {
    cjob_t *c = (cjob_t *)vctx;
    return orc_compress_block(c->p, c->in, c->blk_first[b], c->blk_first[b + 1] - c->blk_first[b],
                              &c->blk_out[b], &c->blk_crc[b], &c->blk_stats[b]);
}

/* get_model_ranking  idn/model_chooser.rs:103-138 (quality 1).  Stable sorts (itertools sorted_by_key). */
static void rank_models(const orc_params_t *p, int type, const orc_reads_t *in, uint64_t n_first,
                        uint32_t model_num, uint32_t *out_idx, uint32_t *out_n) {
    uint32_t idx[256], score[256], n = 0;
    for (uint32_t k = 0; k < p->n_models; k++)
        if (p->models[k]->type == type) {
            idx[n] = k;
            score[n] = 0;
            n++;
        }
    if (n <= 1) { /* model_chooser.rs:37-40 */
        *out_n = n;
        if (n) out_idx[0] = idx[0];
        return;
    }
    for (uint64_t r = 0; r < n_first; r++) {
        size_t len[256];
        uint32_t ord[256];
        uint32_t L = (uint32_t)(in->read_off[r + 1] - in->read_off[r]);
        for (uint32_t k = 0; k < n; k++) {
            len[k] = orc_score_read(p->models[idx[k]], in->acids + in->read_off[r], in->quals + in->read_off[r], L);
            ord[k] = k;
        }
        for (uint32_t a = 1; a < n; a++) /* stable insertion sort by len */
            for (uint32_t b = a; b > 0 && len[ord[b]] < len[ord[b - 1]]; b--) {
                uint32_t t = ord[b];
                ord[b] = ord[b - 1];
                ord[b - 1] = t;
            }
        for (uint32_t i = 0; i < n; i++) score[ord[i]] += i + 1;
    }
    uint32_t ord[256];
    for (uint32_t k = 0; k < n; k++) ord[k] = k;
    for (uint32_t a = 1; a < n; a++)
        for (uint32_t b = a; b > 0 && score[ord[b]] < score[ord[b - 1]]; b--) {
            uint32_t t = ord[b];
            ord[b] = ord[b - 1];
            ord[b - 1] = t;
        }
    *out_n = n < model_num ? n : model_num;
    for (uint32_t i = 0; i < *out_n; i++) out_idx[i] = idx[ord[i]];
}

int orc_compress(const orc_params_t *p_in, const orc_reads_t *in, orc_buf_t *out, orc_stats_t *stats) {
    orc_params_t p = *p_in;
    uint64_t max_len = p.max_block_total_len ? p.max_block_total_len : 4u * 1024 * 1024;
    /* block forming: add_sequence idn/compressor.rs:517-544 */
    uint64_t *first = (uint64_t *)malloc(sizeof(uint64_t) * (in->n_reads + 3));
    uint64_t nb = 0, blen = 0;
    first[0] = 0;
    for (uint64_t r = 0; r < in->n_reads; r++) {
        uint64_t L = in->read_off[r + 1] - in->read_off[r];
        if (L > max_len / 2) {
            free(first);
            return fail(ORC_E_SEQUENCE_TOO_LONG, "sequence too long (%llu > %llu)", (unsigned long long)L,
                        (unsigned long long)(max_len / 2));
        }
        if (blen + L > max_len) {
            first[++nb] = r;
            blen = 0;
        }
        blen += L;
    }
    if (in->n_reads > first[nb]) first[++nb] = in->n_reads; /* finish(): flush partial block :575-578 */
    /* CompressorInitializer  idn/compressor_initializer.rs:33-74 */
    const orc_model_t *retained[256];
    uint32_t n_ret = 0;
    {
        uint32_t model_num = ((uint32_t)p.quality + 1) / 2;
        uint64_t n_first = nb ? first[1] : 0;
        for (int type = 0; type < 2; type++) {
            uint32_t idx[256], n = 0;
            if (p.quality == 1 && !p.fast) {
                rank_models(&p, type, in, n_first, model_num, idx, &n);
            } else {
                /* quality >= 2 uses seeded clustering (clustering.rs:21-118, unpinned RNG): the caller
                 * passes the already-retained list; it is kept in provider order, acids first. */
                for (uint32_t k = 0; k < p.n_models; k++)
                    if (p.models[k]->type == type) idx[n++] = k;
            }
            if (n == 0) {
                free(first);
                return fail(ORC_E_INVALID_STATE, "no %s model registered", type ? "quality score" : "acid");
            }
            for (uint32_t i = 0; i < n; i++) retained[n_ret++] = p.models[idx[i]];
        }
    }
    p.models = retained;
    p.n_models = n_ret;
    /* header + metadata  writer_idn.rs:25-59, data.rs:3-33 */
    buf_put(out, "IDENCOMP", 8);
    buf_u8(out, 1);
    buf_u8(out, 1);
    buf_u8(out, 0);
    buf_u8(out, (uint8_t)n_ret);
    for (uint32_t k = 0; k < n_ret; k++) buf_put(out, retained[k]->id, 32);

    cjob_t c;
    c.p = &p;
    c.in = in;
    c.blk_first = first;
    c.blk_out = (orc_buf_t *)calloc(nb + 1, sizeof(orc_buf_t));
    c.blk_crc = (uint32_t *)calloc(nb + 1, sizeof(uint32_t));
    c.blk_stats = (orc_stats_t *)calloc(nb + 1, sizeof(orc_stats_t));
    int rc = pool_run(p.threads, nb, compress_one, &c);
    if (rc == ORC_OK) {
        for (uint64_t b = 0; b < nb; b++) {
            buf_u32be(out, (uint32_t)c.blk_out[b].len); /* IdnBlockHeader data.rs:35-41 */
            buf_u32be(out, c.blk_crc[b]);
            buf_put(out, c.blk_out[b].data, c.blk_out[b].len);
            if (stats) {
                stats->n_blocks++;
                stats->acid_switches += c.blk_stats[b].acid_switches;
                stats->q_switches += c.blk_stats[b].q_switches;
                stats->out_acid_bytes += c.blk_stats[b].out_acid_bytes;
                stats->out_q_score_bytes += c.blk_stats[b].out_q_score_bytes;
                stats->names_bytes += c.blk_stats[b].names_bytes;
            }
        }
        buf_u32be(out, 0); /* terminator: empty block  idn/compressor.rs:579 */
        buf_u32be(out, 0);
    }
    for (uint64_t b = 0; b < nb; b++) orc_buf_free(&c.blk_out[b]);
    free(c.blk_out);
    free(c.blk_crc);
    free(c.blk_stats);
    free(first);
    return rc;
}

/* ------------------------------------------------------------------------------------------------
 * whole-file decompress
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    uint64_t n_reads, total_len;
    orc_buf_t read_len; /* u32 per read */
    orc_buf_t acids, quals;
    orc_buf_t name_len; /* u32 per read */
    orc_buf_t names;
} blk_dec_t;

typedef struct {
    const orc_model_t *const *models;
    uint32_t n_models;
    const uint8_t *idn;
    const uint64_t *blk_off; /* payload start */
    const uint32_t *blk_len, *blk_crc;
    blk_dec_t *out;
} djob_t;

static uint32_t rd_u32be(const uint8_t *p) {
    return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | (uint32_t)p[3];
}

/* IdnBlockDecompressor::process  idn/decompressor_block.rs:77-239 */
static int decompress_one(void *vctx, uint64_t b) {
    djob_t *d = (djob_t *)vctx;
    const uint8_t *p = d->idn + d->blk_off[b];
    size_t n = d->blk_len[b], pos = 0;
    blk_dec_t *o = &d->out[b];
    int cur_a = -1, cur_q = -1;
    uint32_t crc = 0;
    orc_buf_t names = {0};
    size_t name_pos = 0; /* identifiers are consumed in order (reverse + pop :194-196) */
    int have_names = 0;
    int rc = ORC_OK;
    while (pos < n) {
        uint8_t kind = p[pos++];
        if (kind == 0x00) { /* handle_identifiers_slice :146-163 */
            if (pos + 5 > n) { rc = fail(ORC_E_SERIALIZE, "truncated identifiers header"); break; }
            uint32_t len = rd_u32be(p + pos);
            uint8_t comp = p[pos + 4];
            pos += 5;
            if (pos + len > n) { rc = fail(ORC_E_SERIALIZE, "identifiers slice out of bounds"); break; }
            names.len = 0;
            name_pos = 0;
            if (comp == 1) {
                rc = inflate_names(p + pos, len, &names);
                if (rc) break;
            } else {
                rc = fail(ORC_E_UNSUPPORTED, "Brotli name slices are not restated");
                break;
            }
            have_names = 1;
            pos += len;
        } else if (kind == 0x01) { /* handle_switch_model_slice :194-214 */
            if (pos + 1 > n) { rc = fail(ORC_E_SERIALIZE, "truncated switch slice"); break; }
            uint8_t idx = p[pos++];
            if (idx >= d->n_models) {
                rc = fail(ORC_E_INVALID_MODEL_INDEX, "invalid model index %u (models: %u)", idx, d->n_models);
                break;
            }
            if (d->models[idx]->type == ORC_TYPE_ACID) cur_a = idx; else cur_q = idx;
        } else if (kind == 0x02) { /* handle_sequence_slice :216-239 */
            if (pos + 8 > n) { rc = fail(ORC_E_SERIALIZE, "truncated sequence header"); break; }
            uint32_t len = rd_u32be(p + pos), seq_len = rd_u32be(p + pos + 4);
            pos += 8;
            if (pos + len > n) { rc = fail(ORC_E_SERIALIZE, "sequence slice out of bounds"); break; }
            if (cur_a < 0) { rc = fail(ORC_E_NO_ACTIVE_MODEL, "no active acid model"); break; }
            if (cur_q < 0) { rc = fail(ORC_E_NO_ACTIVE_MODEL, "no active quality score model"); break; }
            buf_reserve(&o->acids, seq_len);
            buf_reserve(&o->quals, seq_len);
            rc = orc_decode_read(d->models[cur_a], d->models[cur_q], p + pos, len, seq_len,
                                 o->acids.data + o->acids.len, o->quals.data + o->quals.len, NULL, NULL);
            if (rc) break;
            /* attach identifier (lines(): split on \n, strip one trailing \r) */
            uint32_t nlen = 0;
            if (have_names && name_pos < names.len) {
                size_t e = name_pos;
                while (e < names.len && names.data[e] != '\n') e++;
                size_t stop = e;
                if (stop > name_pos && names.data[stop - 1] == '\r') stop--;
                nlen = (uint32_t)(stop - name_pos);
                buf_put(&o->names, names.data + name_pos, nlen);
                name_pos = e + 1;
            }
            buf_put(&o->name_len, &nlen, 4);
            crc = orc_crc32(crc, o->names.data + o->names.len - nlen, nlen);
            crc = orc_crc32(crc, o->acids.data + o->acids.len, seq_len);
            crc = orc_crc32(crc, o->quals.data + o->quals.len, seq_len);
            o->acids.len += seq_len;
            o->quals.len += seq_len;
            buf_put(&o->read_len, &seq_len, 4);
            o->n_reads++;
            o->total_len += seq_len;
            pos += len;
        } else {
            rc = fail(ORC_E_SERIALIZE, "unknown slice kind %u", kind);
            break;
        }
    }
    orc_buf_free(&names);
    if (rc == ORC_OK && crc != d->blk_crc[b]) /* check_checksum :131-144 */
        rc = fail(ORC_E_CHECKSUM, "block checksum mismatch (computed %08x, expected %08x)", crc, d->blk_crc[b]);
    return rc;
}

void orc_decoded_free(orc_decoded_t *d) {
    free(d->read_off);
    free(d->acids);
    free(d->quals);
    free(d->name_off);
    free(d->names);
    memset(d, 0, sizeof *d);
}

int orc_decompress(const orc_model_t *const *models, uint32_t n_models, const uint8_t *idn, size_t n,
                   int threads, orc_decoded_t *out) {
    memset(out, 0, sizeof *out);
    size_t pos = 0;
    /* read_header  idn/decompressor.rs:314-322 */
    if (n < 10 || memcmp(idn, "IDENCOMP", 8) != 0) return fail(ORC_E_SERIALIZE, "bad magic");
    out->version = idn[8];
    if (idn[8] != 1) return fail(ORC_E_INVALID_VERSION, "invalid version %u", idn[8]);
    pos = 9;
    /* read_metadata :324-374 */
    uint8_t items = idn[pos++];
    const orc_model_t *sel[256];
    uint32_t n_sel = 0;
    for (uint8_t it = 0; it < items; it++) {
        if (pos + 2 > n) return fail(ORC_E_SERIALIZE, "truncated metadata");
        uint8_t magic = idn[pos++];
        if (magic != 0) return fail(ORC_E_SERIALIZE, "unknown metadata item %u", magic);
        uint8_t nm = idn[pos++];
        if (pos + 32u * nm > n) return fail(ORC_E_SERIALIZE, "truncated model list");
        n_sel = 0;
        for (uint8_t k = 0; k < nm; k++) {
            const uint8_t *id = idn + pos + 32u * k;
            memcpy(out->model_ids[k], id, 32);
            const orc_model_t *found = NULL;
            for (uint32_t j = 0; j < n_models; j++)
                if (memcmp(models[j]->id, id, 32) == 0) {
                    found = models[j];
                    break;
                }
            if (!found) return fail(ORC_E_UNKNOWN_MODEL, "unknown model %02x%02x%02x%02x", id[0], id[1], id[2], id[3]);
            sel[n_sel++] = found; /* filter_by_identifiers  model_provider.rs:290-329 */
        }
        out->n_models = nm;
        pos += 32u * nm;
    }
    /* block index */
    size_t cap = 16, nb = 0;
    uint64_t *off = (uint64_t *)malloc(cap * sizeof(uint64_t));
    uint32_t *len = (uint32_t *)malloc(cap * sizeof(uint32_t));
    uint32_t *crc = (uint32_t *)malloc(cap * sizeof(uint32_t));
    int rc = ORC_OK;
    for (;;) { /* read_next_block :387-428 */
        if (pos + 8 > n) { rc = fail(ORC_E_IO, "unexpected end of file in block header"); break; }
        uint32_t l = rd_u32be(idn + pos), c = rd_u32be(idn + pos + 4);
        pos += 8;
        if (pos + l > n) { rc = fail(ORC_E_IO, "unexpected end of file in block"); break; }
        if (nb == cap) {
            cap *= 2;
            off = (uint64_t *)realloc(off, cap * sizeof(uint64_t));
            len = (uint32_t *)realloc(len, cap * sizeof(uint32_t));
            crc = (uint32_t *)realloc(crc, cap * sizeof(uint32_t));
        }
        off[nb] = pos;
        len[nb] = l;
        crc[nb] = c;
        nb++;
        pos += l;
        if (l == 0) break; /* EOF marker */
    }
    blk_dec_t *bo = (blk_dec_t *)calloc(nb ? nb : 1, sizeof(blk_dec_t));
    if (rc == ORC_OK) {
        djob_t d = {sel, n_sel, idn, off, len, crc, bo};
        rc = pool_run(threads, nb, decompress_one, &d);
    }
    if (rc == ORC_OK) {
        uint64_t R = 0, T = 0, NB = 0;
        for (size_t b = 0; b < nb; b++) {
            R += bo[b].n_reads;
            T += bo[b].total_len;
            NB += bo[b].names.len;
        }
        out->n_reads = R;
        out->total_len = T;
        out->n_blocks = nb;
        out->read_off = (uint64_t *)malloc((R + 1) * sizeof(uint64_t));
        out->name_off = (uint64_t *)malloc((R + 1) * sizeof(uint64_t));
        out->acids = (uint8_t *)malloc(T + 1);
        out->quals = (uint8_t *)malloc(T + 1);
        out->names = (uint8_t *)malloc(NB + 1);
        uint64_t r = 0, t = 0, nn = 0;
        out->read_off[0] = 0;
        out->name_off[0] = 0;
        for (size_t b = 0; b < nb; b++) {
            memcpy(out->acids + t, bo[b].acids.data, bo[b].total_len);
            memcpy(out->quals + t, bo[b].quals.data, bo[b].total_len);
            memcpy(out->names + nn, bo[b].names.data, bo[b].names.len);
            const uint32_t *rl = (const uint32_t *)bo[b].read_len.data;
            const uint32_t *nl = (const uint32_t *)bo[b].name_len.data;
            for (uint64_t k = 0; k < bo[b].n_reads; k++) {
                t += rl[k];
                nn += nl[k];
                r++;
                out->read_off[r] = t;
                out->name_off[r] = nn;
            }
        }
    }
    for (size_t b = 0; b < nb; b++) {
        orc_buf_free(&bo[b].read_len);
        orc_buf_free(&bo[b].acids);
        orc_buf_free(&bo[b].quals);
        orc_buf_free(&bo[b].name_len);
        orc_buf_free(&bo[b].names);
    }
    free(bo);
    free(off);
    free(len);
    free(crc);
    return rc;
}

/* ------------------------------------------------------------------------------------------------
 * FASTQ text (fastq/reader.rs:166-282, consts.rs:28-98, writer.rs:190-240) -- host-side, out of the GPU
 * path; here so the goldens (samples/*.fastq) can be turned into symbol arrays, and as the statement the
 * device reader's acceptance and error reports are checked against.
 *
 * A record is checked in the reference's order: the title starts with '@' (untrimmed line), the acids
 * line is present, every acid is valid, the separator line is present and starts with '+', the quality
 * line is present, every byte of the whole quality line is valid, and only then are the two lengths
 * compared.  A missing line is EofReached.  Blank lines (ASCII white space only: 0x09-0x0D and ' ', as
 * str::trim does for ASCII) are skipped where a title is expected, and the title is trimmed with the same
 * set.  A failure is reported as "FastqReaderError::<variant> at record <r>", r counted from 0 in file
 * order; oracle.py parses that form.
 * ---------------------------------------------------------------------------------------------- */
static const uint8_t *next_line(const uint8_t *p, const uint8_t *end, const uint8_t **ls, const uint8_t **le) {
    if (p >= end) return NULL;
    const uint8_t *nl = (const uint8_t *)memchr(p, '\n', (size_t)(end - p));
    *ls = p;
    *le = nl ? nl : end;
    return nl ? nl + 1 : end;
}

static int fq_ws(uint8_t c) { return c == ' ' || (c >= 9 && c <= 13); }

static int fq_fail(const char *variant, uint64_t record) {
    return fail(ORC_E_FASTQ, "FastqReaderError::%s at record %llu", variant, (unsigned long long)record);
}

int orc_fastq_parse(const uint8_t *text, size_t n, orc_decoded_t *out) {
    memset(out, 0, sizeof *out);
    orc_buf_t ro = {0}, no = {0}, ac = {0}, qu = {0}, nm = {0};
    uint64_t z = 0;
    buf_put(&ro, &z, 8);
    buf_put(&no, &z, 8);
    const uint8_t *p = text, *end = text + n, *ls, *le;
    int rc = ORC_OK;
    for (;;) {
        const uint64_t rec = out->n_reads;
        /* parse_title: skip blank lines, require '@', trim */
        const uint8_t *q;
        int got = 0;
        while ((q = next_line(p, end, &ls, &le)) != NULL) {
            p = q;
            const uint8_t *a = ls, *b = le;
            while (a < b && fq_ws(*a)) a++;
            if (a < b) {
                got = 1;
                break;
            }
        }
        if (!got) break; /* EOF */
        if (*ls != '@') { rc = fq_fail("InvalidFormat", rec); break; }
        const uint8_t *a = ls + 1, *b = le;
        while (a < b && fq_ws(*a)) a++;
        while (b > a && fq_ws(b[-1])) b--;
        buf_put(&nm, a, (size_t)(b - a));
        /* acids */
        if ((q = next_line(p, end, &ls, &le)) == NULL) { rc = fq_fail("EofReached", rec); break; }
        p = q;
        size_t alen = (size_t)(le - ls);
        buf_reserve(&ac, alen);
        for (size_t i = 0; i < alen && !rc; i++) {
            uint8_t v;
            switch (ls[i]) { /* Acid repr: N=0 A=1 C=2 T=3 G=4  sequence.rs:401-413 */
            case 'N': v = 0; break;
            case 'A': v = 1; break;
            case 'C': v = 2; break;
            case 'T': v = 3; break;
            case 'G': v = 4; break;
            default: rc = fq_fail("InvalidAcid", rec); v = 0;
            }
            ac.data[ac.len + i] = v;
        }
        if (rc) break;
        ac.len += alen;
        /* separator */
        if ((q = next_line(p, end, &ls, &le)) == NULL) { rc = fq_fail("EofReached", rec); break; }
        p = q;
        if (le == ls || *ls != '+') { rc = fq_fail("InvalidFormat", rec); break; }
        /* quality scores: the whole line is converted before the lengths are compared */
        if ((q = next_line(p, end, &ls, &le)) == NULL) { rc = fq_fail("EofReached", rec); break; }
        p = q;
        size_t qlen = (size_t)(le - ls);
        buf_reserve(&qu, qlen);
        for (size_t i = 0; i < qlen; i++) {
            uint8_t ch = ls[i];
            if (ch < '!' || ch > '~') { rc = fq_fail("InvalidQualityScore", rec); break; }
            qu.data[qu.len + i] = (uint8_t)(ch - '!');
        }
        if (rc) break;
        if (qlen != alen) { rc = fq_fail("AcidAndQualityScoreLengthMismatch", rec); break; }
        qu.len += qlen;
        uint64_t t = ac.len, nn = nm.len;
        buf_put(&ro, &t, 8);
        buf_put(&no, &nn, 8);
        out->n_reads++;
    }
    if (rc) {
        orc_buf_free(&ro); orc_buf_free(&no); orc_buf_free(&ac); orc_buf_free(&qu); orc_buf_free(&nm);
        return rc;
    }
    out->total_len = ac.len;
    out->read_off = (uint64_t *)ro.data;
    out->name_off = (uint64_t *)no.data;
    buf_reserve(&ac, 1); buf_reserve(&qu, 1); buf_reserve(&nm, 1);
    out->acids = ac.data;
    out->quals = qu.data;
    out->names = nm.data;
    return ORC_OK;
}

int orc_fastq_write(const orc_reads_t *in, orc_buf_t *out) {
    static const char A2B[5] = {'N', 'A', 'C', 'T', 'G'};
    for (uint64_t r = 0; r < in->n_reads; r++) {
        uint64_t L = in->read_off[r + 1] - in->read_off[r];
        buf_u8(out, '@');
        if (in->name_off) buf_put(out, in->names + in->name_off[r], in->name_off[r + 1] - in->name_off[r]);
        buf_u8(out, '\n');
        buf_reserve(out, 2 * L + 4);
        for (uint64_t i = 0; i < L; i++) out->data[out->len + i] = (uint8_t)A2B[in->acids[in->read_off[r] + i]];
        out->len += L;
        buf_put(out, "\n+\n", 3);
        for (uint64_t i = 0; i < L; i++) out->data[out->len + i] = (uint8_t)(in->quals[in->read_off[r] + i] + '!');
        out->len += L;
        buf_u8(out, '\n');
    }
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------------
 * Workload generator (bench/test utility; SURVEY.md 8d): model-driven synthetic reads.  Restates the
 * sampler of the device library's workload generator so that the CPU baseline and the GPU path can be
 * fed identical inputs without copying between them: SplitMix64 keyed by (seed, read index), one draw
 * per position: acid slot = bits 0..13, q slot = bits 14..27, N-injection = (bits 32..63) % 1e6 < n_ppm.
 * ---------------------------------------------------------------------------------------------- */
static uint64_t splitmix64(uint64_t *s) {
    uint64_t z = (*s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

static uint32_t sym_for_slot(const orc_model_t *m, uint32_t row, uint32_t slot) {
    const uint16_t *c = m->cum + (size_t)row * (m->nsym + 1);
    uint32_t lo = 0, hi = m->nsym; /* largest s with c[s] <= slot */
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) / 2;
        if (c[mid] <= slot) lo = mid; else hi = mid;
    }
    return lo;
}

typedef struct {
    const orc_model_t *am, *qm;
    const uint64_t *read_off;
    uint64_t n_reads, first_read_index, seed;
    uint32_t n_ppm;
    uint8_t *acids, *quals;
} synth_job_t;

static int synth_chunk(void *vc, uint64_t chunk) {
    synth_job_t *j = (synth_job_t *)vc;
    uint64_t r0 = chunk * 4096, r1 = r0 + 4096;
    if (r1 > j->n_reads) r1 = j->n_reads;
    for (uint64_t r = r0; r < r1; r++) {
        uint64_t off = j->read_off[r];
        uint32_t len = (uint32_t)(j->read_off[r + 1] - off);
        uint64_t s = j->seed ^ ((j->first_read_index + r + 1) * 0xD1B54A32D192ED03ull);
        orc_gen_t ga, gq;
        orc_gen_init(&ga, &j->am->spec, len);
        orc_gen_init(&gq, &j->qm->spec, len);
        uint32_t prev_q = 0;
        for (uint32_t i = 0; i < len; i++) {
            uint64_t u = splitmix64(&s);
            uint32_t slot_a = (uint32_t)u & 0x3fffu, slot_q = (uint32_t)(u >> 14) & 0x3fffu;
            uint32_t row_a = ctx_for(j->am, orc_gen_current(&ga)), row_q = ctx_for(j->qm, orc_gen_current(&gq));
            uint32_t a = sym_for_slot(j->am, row_a, slot_a);
            uint32_t q = sym_for_slot(j->qm, row_q, slot_q);
            /* unseen context (dummy row): plain base / previous quality score, see the device sampler */
            if (row_a == 0) a = 1 + (slot_a & 3u);
            if (row_q == 0 && i > 0) q = prev_q;
            if ((uint32_t)((u >> 32) % 1000000u) < j->n_ppm) {
                a = 0;
                q = 2;
            }
            prev_q = q;
            j->acids[off + i] = (uint8_t)a;
            j->quals[off + i] = (uint8_t)q;
            orc_gen_update(&ga, (uint8_t)a, (uint8_t)q);
            orc_gen_update(&gq, (uint8_t)a, (uint8_t)q);
        }
    }
    return 0;
}

int orc_synth_reads(const orc_model_t *am, const orc_model_t *qm, const uint64_t *read_off, uint64_t n_reads,
                    uint64_t first_read_index, uint64_t seed, uint32_t n_ppm, int threads, uint8_t *acids,
                    uint8_t *quals) {
    if (am->type != ORC_TYPE_ACID || qm->type != ORC_TYPE_QSCORE)
        return fail(ORC_E_INVALID_STATE, "need an acid model and a quality score model");
    synth_job_t j = {am, qm, read_off, n_reads, first_read_index, seed, n_ppm, acids, quals};
    return pool_run(threads, (n_reads + 4095) / 4096, synth_chunk, &j);
}

/* ------------------------------------------------------------------------------------------------
 * GPU-native multi-lane block format (container version 2).  NOT part of the reference: this is an
 * independent CPU statement of the format specified in DESIGN.md section 8 (and in the header of
 * idencomp_b200/csrc/idn_native.cuh), used to check the CUDA encoder/decoder of that format bit for bit.
 * It reuses the pinned per-symbol machinery above (generators, tables, ryg put/get); only stream
 * segmentation and framing are new.
 * ---------------------------------------------------------------------------------------------- */
#define NATIVE_HDR_FIXED 22u

static void put_u32be(uint8_t *p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24);
    p[1] = (uint8_t)(v >> 16);
    p[2] = (uint8_t)(v >> 8);
    p[3] = (uint8_t)v;
}
static uint32_t get_u32be(const uint8_t *p) {
    return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3];
}

/* Lane partition of a block (normative text: idencomp_b200/csrc/idn_native.cuh).
 *   pieces: a read of length L is ONE piece, unless lane_syms >= 256 and L > lane_syms: then it is cut into
 *           ceil(L / lane_syms) pieces of lane_syms symbols (the last one shorter);
 *   lanes:  with o_p the block-relative offset of the first symbol of piece p, a new lane starts at the first piece of the
 *           block and at every piece with o_p / lane_syms != o_(p-1) / lane_syms.
 * A lane is therefore a contiguous range of the block's symbol stream; empty reads carry no symbols and do not matter.
 * Returns the lane start offsets (block-relative) in lane_sym[0 .. n_lanes], lane_sym[n_lanes] = block symbols. */
#define NATIVE_MIN_SPLIT_Q 256u
#define NATIVE_HIST 8u
static uint64_t native_lanes(const uint32_t *lens, uint64_t n_reads, uint32_t Q, uint64_t *lane_sym, int *split_out) {
    uint64_t n_lanes = 0, off = 0, prev_q = 0;
    int first = 1, split = 0;
    for (uint64_t i = 0; i < n_reads; i++) {
        const uint32_t len = lens[i];
        const uint64_t pc = (Q >= NATIVE_MIN_SPLIT_Q && len > Q) ? ((uint64_t)len + Q - 1) / Q : 1;
        if (pc > 1) split = 1;
        for (uint64_t j = 0; j < pc; j++) {
            const uint64_t o = off + j * Q;
            if (first || o / Q != prev_q) lane_sym[n_lanes++] = o;
            first = 0;
            prev_q = o / Q;
        }
        off += len;
    }
    lane_sym[n_lanes] = off;
    if (split_out) *split_out = split;
    return n_lanes;
}

/* one lane = the symbols [a, b) of the block's stream, pushed last -> first onto one 2-state stream: every read is walked
 * by its generators from its first position (the contexts of a piece that starts inside a read are the true ones);
 * returns the payload length */
static size_t native_encode_lane(const orc_model_t *am, const orc_model_t *qm, const orc_reads_t *in, uint64_t first_read,
                                 uint64_t n_reads, uint64_t a, uint64_t b, uint8_t *tmp, size_t cap, uint8_t **start_out) {
    uint32_t s0 = RANS_L, s1 = RANS_L;
    uint8_t *ptr = tmp + cap;
    const uint64_t base = in->read_off[first_read];
    for (uint64_t r = first_read + n_reads; r-- > first_read;) {
        const uint64_t ro = in->read_off[r] - base, re = in->read_off[r + 1] - base;
        if (ro >= b || re <= a) continue;
        const uint32_t len = (uint32_t)(re - ro);
        const uint32_t p0 = (uint32_t)((a > ro ? a : ro) - ro), p1 = (uint32_t)((b < re ? b : re) - ro);
        const uint8_t *ac = in->acids + in->read_off[r];
        const uint8_t *qu = in->quals + in->read_off[r];
        uint32_t *ctx_a = (uint32_t *)malloc(((size_t)p1 + 1) * 2 * sizeof(uint32_t));
        uint32_t *ctx_q = ctx_a + p1 + 1;
        orc_gen_t ga, gq;
        orc_gen_init(&ga, &am->spec, len);
        orc_gen_init(&gq, &qm->spec, len);
        for (uint32_t i = 0; i < p1; i++) {
            ctx_a[i] = ctx_for(am, orc_gen_current(&ga));
            ctx_q[i] = ctx_for(qm, orc_gen_current(&gq));
            orc_gen_update(&ga, ac[i], qu[i]);
            orc_gen_update(&gq, ac[i], qu[i]);
        }
        for (uint32_t i = p1; i-- > p0;) {
            enc_put(&s0, &ptr, &am->enc[(size_t)ctx_a[i] * ORC_ACID_SYMS + ac[i]]);
            enc_put(&s1, &ptr, &qm->enc[(size_t)ctx_q[i] * ORC_Q_SYMS + qu[i]]);
        }
        free(ctx_a);
    }
    enc_flush(s0, &ptr);
    enc_flush(s1, &ptr);
    *start_out = ptr;
    return (size_t)(tmp + cap - ptr);
}

/* slices of one version-2 block (no block header): [Identifiers] NativeLanes; crc as in version 1 */
int orc_compress_native_block(const orc_params_t *p, const orc_reads_t *in, uint64_t first_read, uint64_t n_reads,
                              uint32_t lane_syms, orc_buf_t *out, uint32_t *crc_out) {
    uint32_t crc = 0;
    *crc_out = 0;
    if (n_reads == 0) return ORC_OK;
    if (lane_syms == 0) return fail(ORC_E_INVALID_STATE, "lane_syms must be positive");
    if (p->include_identifiers) {
        orc_buf_t joined = {0}, z = {0};
        for (uint64_t r = first_read; r < first_read + n_reads; r++) {
            if (r > first_read) buf_u8(&joined, '\n');
            if (in->name_off) buf_put(&joined, in->names + in->name_off[r], in->name_off[r + 1] - in->name_off[r]);
        }
        int rc = deflate_names(joined.data, joined.len, p->deflate_level ? p->deflate_level : 6, &z);
        if (rc) {
            orc_buf_free(&joined);
            orc_buf_free(&z);
            return rc;
        }
        buf_u8(out, 0x00);
        buf_u32be(out, (uint32_t)z.len);
        buf_u8(out, 1);
        buf_put(out, z.data, z.len);
        orc_buf_free(&joined);
        orc_buf_free(&z);
    }
    /* candidates per type in provider order */
    int cand[2][256], n_cand[2] = {0, 0};
    for (uint32_t k = 0; k < p->n_models; k++) cand[p->models[k]->type][n_cand[p->models[k]->type]++] = (int)k;
    if (!n_cand[0] || !n_cand[1]) return fail(ORC_E_INVALID_STATE, "need at least one model per type");
    /* lane partition */
    const uint64_t base = in->read_off[first_read];
    const uint64_t n_syms = in->read_off[first_read + n_reads] - base;
    uint32_t *lens = (uint32_t *)malloc(sizeof(uint32_t) * (n_reads + 1));
    uint32_t mn = 0xffffffffu, mx = 0;
    for (uint64_t i = 0; i < n_reads; i++) {
        lens[i] = (uint32_t)(in->read_off[first_read + i + 1] - in->read_off[first_read + i]);
        if (lens[i] < mn) mn = lens[i];
        if (lens[i] > mx) mx = lens[i];
    }
    uint64_t *lane_sym = (uint64_t *)malloc(sizeof(uint64_t) * (n_reads + n_syms / lane_syms + 2));
    int split = 0;
    const uint64_t n_lanes = native_lanes(lens, n_reads, lane_syms, lane_sym, &split);
    uint32_t width = mn == mx ? 0u : (mx < 65536u ? 2u : 4u);
    /* per-lane model choice and payloads */
    uint8_t *mdl = (uint8_t *)malloc(2 * n_lanes + 2);
    uint32_t *llen = (uint32_t *)malloc(sizeof(uint32_t) * (n_lanes + 1));
    uint64_t *score = NULL;
    if ((n_cand[0] > 1 || n_cand[1] > 1) && !p->fast) { /* forward scores of every read under every model, computed once */
        score = (uint64_t *)malloc(sizeof(uint64_t) * n_reads * p->n_models);
        for (uint64_t i = 0; i < n_reads; i++)
            for (uint32_t k = 0; k < p->n_models; k++)
                score[i * p->n_models + k] = orc_score_read(p->models[k], in->acids + in->read_off[first_read + i],
                                                            in->quals + in->read_off[first_read + i], lens[i]);
    }
    orc_buf_t pay = {0};
    uint64_t r_lo = 0; /* first read with a symbol at or behind the start of the current lane */
    for (uint64_t l = 0; l < n_lanes; l++) {
        const uint64_t a = lane_sym[l], b = lane_sym[l + 1];
        while (r_lo < n_reads && in->read_off[first_read + r_lo + 1] - base <= a) r_lo++;
        int pick[2];
        for (int type = 0; type < 2; type++) {
            pick[type] = cand[type][0];
            if (n_cand[type] > 1 && !p->fast) {
                /* argmin over the candidates of the summed forward scores of the reads with at least one symbol in the lane */
                uint64_t best = ~0ull;
                for (int k = 0; k < n_cand[type]; k++) {
                    uint64_t sum = 0;
                    for (uint64_t i = r_lo; i < n_reads && in->read_off[first_read + i] - base < b; i++)
                        if (in->read_off[first_read + i + 1] - base > a) sum += score[i * p->n_models + cand[type][k]];
                    if (sum < best) { /* first minimum wins */
                        best = sum;
                        pick[type] = cand[type][k];
                    }
                }
            }
        }
        mdl[2 * l] = (uint8_t)pick[0];
        mdl[2 * l + 1] = (uint8_t)pick[1];
        /* a lane that starts inside a read carries the (acid, quality score) pairs of the NATIVE_HIST positions in front of it
         * (zeros before the start of the read): the decoder rebuilds the generator states from them */
        const uint64_t rr = r_lo;
        const int mid = rr < n_reads && in->read_off[first_read + rr] - base < a && b > a;
        size_t cap = 4 * (size_t)(b - a) + 8;
        uint8_t *tmp = (uint8_t *)malloc(cap), *start;
        size_t n = native_encode_lane(p->models[pick[0]], p->models[pick[1]], in, first_read, n_reads, a, b, tmp, cap, &start);
        if (mid) {
            uint8_t hist[2 * NATIVE_HIST];
            const uint64_t ro = in->read_off[first_read + rr] - base;
            for (uint32_t k = 0; k < NATIVE_HIST; k++) {
                const uint64_t pos = a - NATIVE_HIST + k; /* block-relative */
                const int inside = a >= NATIVE_HIST - k + ro && pos >= ro;
                hist[k] = inside ? in->acids[base + pos] : 0;
                hist[NATIVE_HIST + k] = inside ? in->quals[base + pos] : 0;
            }
            buf_put(&pay, hist, sizeof hist);
        }
        llen[l] = (uint32_t)(n + (mid ? 2 * NATIVE_HIST : 0));
        buf_put(&pay, start, n);
        free(tmp);
    }
    for (uint64_t r = first_read; r < first_read + n_reads; r++) {
        uint32_t len = (uint32_t)(in->read_off[r + 1] - in->read_off[r]);
        if (in->name_off && p->include_identifiers)
            crc = orc_crc32(crc, in->names + in->name_off[r], in->name_off[r + 1] - in->name_off[r]);
        crc = orc_crc32(crc, in->acids + in->read_off[r], len);
        crc = orc_crc32(crc, in->quals + in->read_off[r], len);
    }
    uint64_t body = NATIVE_HDR_FIXED - 5 + n_reads * width + 6 * n_lanes + pay.len;
    buf_u8(out, 0x03);
    buf_u32be(out, (uint32_t)body);
    buf_u32be(out, (uint32_t)n_reads);
    buf_u32be(out, (uint32_t)n_lanes);
    buf_u32be(out, lane_syms);
    buf_u8(out, (uint8_t)(width | (split ? 0x80u : 0u)));
    buf_u32be(out, width == 0 ? mn : 0);
    for (uint64_t r = first_read; r < first_read + n_reads && width; r++) {
        uint32_t len = (uint32_t)(in->read_off[r + 1] - in->read_off[r]);
        if (width == 2) {
            buf_u8(out, (uint8_t)(len >> 8));
            buf_u8(out, (uint8_t)len);
        } else {
            buf_u32be(out, len);
        }
    }
    buf_put(out, mdl, 2 * n_lanes);
    for (uint64_t l = 0; l < n_lanes; l++) buf_u32be(out, llen[l]);
    buf_put(out, pay.data, pay.len);
    orc_buf_free(&pay);
    free(mdl);
    free(llen);
    free(lane_sym);
    free(lens);
    free(score);
    *crc_out = crc;
    return ORC_OK;
}

/* decode the NativeLanes slice of one version-2 block (Identifiers slices are skipped); outputs are appended to
 * acids/quals at *n_syms and lengths to read_len at *n_reads (capacities are the caller's business: sized from the
 * header fields, which the caller can read with orc_native_block_counts) */
int orc_native_block_counts(const uint8_t *data, size_t n, uint64_t *n_reads, uint64_t *n_syms) {
    size_t pos = 0;
    *n_reads = *n_syms = 0;
    while (pos < n) {
        if (data[pos] == 0) {
            if (pos + 6 > n) return fail(ORC_E_SERIALIZE, "truncated identifiers slice");
            size_t len = get_u32be(data + pos + 1);
            if (len > n - pos - 6) return fail(ORC_E_SERIALIZE, "truncated identifiers slice");
            pos += 6 + len;
        } else if (data[pos] == 3) {
            if (pos + NATIVE_HDR_FIXED > n) return fail(ORC_E_SERIALIZE, "truncated native slice");
            uint32_t body = get_u32be(data + pos + 1), nr = get_u32be(data + pos + 5), w = data[pos + 17] & 0x7fu;
            if (body > n - pos - 5) return fail(ORC_E_SERIALIZE, "truncated native slice");
            *n_reads += nr;
            if (w == 0) {
                *n_syms += (uint64_t)nr * get_u32be(data + pos + 18);
            } else {
                if ((uint64_t)nr * w > body) return fail(ORC_E_SERIALIZE, "bad length table");
                for (uint32_t i = 0; i < nr; i++)
                    *n_syms += w == 2 ? (uint32_t)(data[pos + 22 + 2 * i] << 8 | data[pos + 23 + 2 * i])
                                      : get_u32be(data + pos + 22 + 4 * (size_t)i);
            }
            pos += 5 + (size_t)body;
        } else {
            return fail(ORC_E_SERIALIZE, "unexpected slice kind %u in a version 2 block", data[pos]);
        }
    }
    return ORC_OK;
}

int orc_decompress_native_block(const orc_model_t *const *models, uint32_t n_models, const uint8_t *data, size_t n,
                                uint8_t *acids, uint8_t *quals, uint32_t *read_len) {
    size_t pos = 0;
    uint64_t out_sym = 0, out_read = 0;
    const uint32_t mask = (1u << ORC_SCALE_BITS) - 1;
    while (pos < n) {
        if (data[pos] == 0) {
            pos += 6 + (size_t)get_u32be(data + pos + 1);
            continue;
        }
        if (data[pos] != 3) return fail(ORC_E_SERIALIZE, "unexpected slice kind");
        uint32_t body = get_u32be(data + pos + 1), nr = get_u32be(data + pos + 5), nl = get_u32be(data + pos + 9);
        uint32_t Q = get_u32be(data + pos + 13), w = data[pos + 17] & 0x7fu, cl = get_u32be(data + pos + 18);
        const int split_flag = data[pos + 17] >> 7;
        const uint8_t *t_len = data + pos + NATIVE_HDR_FIXED;
        const uint8_t *t_mdl = t_len + (size_t)nr * w;
        const uint8_t *t_ll = t_mdl + 2 * (size_t)nl;
        const uint8_t *pay = t_ll + 4 * (size_t)nl;
        if (Q == 0 || (size_t)(pay - (data + pos + 5)) > body) return fail(ORC_E_SERIALIZE, "bad native header");
        uint32_t *lens = (uint32_t *)malloc(sizeof(uint32_t) * ((size_t)nr + 1));
        uint64_t *roff = (uint64_t *)malloc(sizeof(uint64_t) * ((size_t)nr + 1));
        uint64_t total = 0;
        for (uint32_t i = 0; i < nr; i++) {
            lens[i] = w == 0 ? cl : (w == 2 ? (uint32_t)(t_len[2 * i] << 8 | t_len[2 * i + 1]) : get_u32be(t_len + 4 * (size_t)i));
            roff[i] = total;
            total += lens[i];
            read_len[out_read++] = lens[i];
        }
        roff[nr] = total;
        uint64_t *lane_sym = (uint64_t *)malloc(sizeof(uint64_t) * ((size_t)nr + total / Q + 2));
        int split = 0;
        const uint64_t n_lanes = nr ? native_lanes(lens, nr, Q, lane_sym, &split) : 0;
        if (n_lanes != nl || split != split_flag) {
            free(lens); free(roff); free(lane_sym);
            return fail(ORC_E_SERIALIZE, "the lane table does not match the partition of the lengths");
        }
        uint32_t r = 0;
        for (uint64_t lane = 0; lane < n_lanes; lane++) {
            const uint64_t a = lane_sym[lane], b = lane_sym[lane + 1];
            uint32_t ia = t_mdl[2 * lane], iq = t_mdl[2 * lane + 1], ll = get_u32be(t_ll + 4 * (size_t)lane);
            if (ia >= n_models || iq >= n_models || models[ia]->type != ORC_TYPE_ACID || models[iq]->type != ORC_TYPE_QSCORE) {
                free(lens); free(roff); free(lane_sym);
                return fail(ORC_E_INVALID_MODEL_INDEX, "lane names a bad model");
            }
            while (r < nr && roff[r + 1] <= a) r++; /* first read with a symbol at or behind a */
            const int mid = r < nr && roff[r] < a && b > a;
            const uint32_t hdr = mid ? 2 * NATIVE_HIST : 0;
            if (ll < 8 + hdr || (size_t)(pay - data) + ll > pos + 5 + (size_t)body) {
                free(lens); free(roff); free(lane_sym);
                return fail(ORC_E_SERIALIZE, "lane payload out of range");
            }
            const orc_model_t *am = models[ia], *qm = models[iq];
            const uint8_t *st = pay + hdr;
            uint32_t sq = (uint32_t)st[0] | (uint32_t)st[1] << 8 | (uint32_t)st[2] << 16 | (uint32_t)st[3] << 24;
            uint32_t sa = (uint32_t)st[4] | (uint32_t)st[5] << 8 | (uint32_t)st[6] << 16 | (uint32_t)st[7] << 24;
            size_t pp = hdr + 8;
            for (uint32_t k = r; k < nr && roff[k] < b; k++) {
                if (roff[k + 1] <= a) continue;
                const uint32_t len = lens[k];
                const uint32_t p0 = (uint32_t)((a > roff[k] ? a : roff[k]) - roff[k]), p1 = (uint32_t)((b < roff[k + 1] ? b : roff[k + 1]) - roff[k]);
                orc_gen_t ga, gq;
                orc_gen_init(&ga, &am->spec, len);
                orc_gen_init(&gq, &qm->spec, len);
                if (p0 > 0) { /* a piece that starts inside its read: states from the stored history, position counter = p0 */
                    ga.position = gq.position = p0 - NATIVE_HIST; /* u32 wrap is undone by the NATIVE_HIST updates below */
                    for (uint32_t h = 0; h < NATIVE_HIST; h++) {
                        orc_gen_update(&ga, pay[h], pay[NATIVE_HIST + h]);
                        orc_gen_update(&gq, pay[h], pay[NATIVE_HIST + h]);
                    }
                }
                for (uint32_t i = p0; i < p1; i++) {
                    uint32_t ca = ctx_for(am, orc_gen_current(&ga)), cq = ctx_for(qm, orc_gen_current(&gq));
                    uint32_t slot_q = sq & mask, slot_a = sa & mask;
                    uint32_t yq = find_sym(qm, cq, slot_q), ya = find_sym(am, ca, slot_a);
                    const uint16_t *rq = qm->cum + (size_t)cq * (ORC_Q_SYMS + 1);
                    const uint16_t *ra = am->cum + (size_t)ca * (ORC_ACID_SYMS + 1);
                    sq = (uint32_t)(rq[yq + 1] - rq[yq]) * (sq >> ORC_SCALE_BITS) + slot_q - rq[yq];
                    sa = (uint32_t)(ra[ya + 1] - ra[ya]) * (sa >> ORC_SCALE_BITS) + slot_a - ra[ya];
                    while (sq < RANS_L) {
                        if (pp >= ll) { free(lens); free(roff); free(lane_sym); return fail(ORC_E_SERIALIZE, "lane payload exhausted"); }
                        sq = (sq << 8) | pay[pp++];
                    }
                    while (sa < RANS_L) {
                        if (pp >= ll) { free(lens); free(roff); free(lane_sym); return fail(ORC_E_SERIALIZE, "lane payload exhausted"); }
                        sa = (sa << 8) | pay[pp++];
                    }
                    acids[out_sym + roff[k] + i] = (uint8_t)ya;
                    quals[out_sym + roff[k] + i] = (uint8_t)yq;
                    orc_gen_update(&ga, (uint8_t)ya, (uint8_t)yq);
                    orc_gen_update(&gq, (uint8_t)ya, (uint8_t)yq);
                }
            }
            if (sq != RANS_L || sa != RANS_L || pp != ll) { free(lens); free(roff); free(lane_sym); return fail(ORC_E_SERIALIZE, "lane does not end cleanly"); }
            pay += ll;
        }
        out_sym += total;
        free(lens);
        free(roff);
        free(lane_sym);
        if ((size_t)(pay - (data + pos + 5)) != body) return fail(ORC_E_SERIALIZE, "native slice framing mismatch");
        pos += 5 + (size_t)body;
    }
    return ORC_OK;
}
