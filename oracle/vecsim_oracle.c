/* vecsim_oracle.c — CPU restatement of the reference's FLAT (brute-force) VecSim path.
 * TEST INFRASTRUCTURE ONLY (see oracle.h).  Pinned against oracle/_ref/libvecsim_ref.so (the
 * reference's own sources) by tests/test_oracle_vecsim.py.
 *
 * Follows, function by function:
 *   distances     VS/spaces/L2/L2.cpp:76-174, VS/spaces/IP/IP.cpp:185-285 (scalar baselines),
 *                 VS/spaces/L2/L2_AVX512F_FP32.h:21-59, VS/spaces/IP/IP_AVX512F_FP32.h:19-56
 *                 (fp32 AVX-512 tier, emulated lane by lane with fmaf)
 *   normalisers   VS/spaces/normalize/normalize_naive.h:23-88, compute_norm.h:17-28
 *   conversions   VS/types/float16.h:33-117, VS/types/bfloat16.h:22-38
 *   index         VS/algorithms/brute_force/brute_force.h:175-451, brute_force_single.h:135-212,
 *                 brute_force_multi.h
 *   heap order    VS/utils/vecsim_stl.h:64-84 (max-heap of pair<float,size_t>, std::less)
 */
#include "oracle.h"

#include <float.h>
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

/* ------------------------------------------------------------------ conversions ------------ */
static inline float u2f(uint32_t u) {
    float f;
    memcpy(&f, &u, 4);
    return f;
}
static inline uint32_t f2u(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}

float orc_half_to_float(uint16_t h) { /* float16.h:33-52 */
    const uint32_t shifted_exp = 0x7c00u << 13;
    int32_t o = ((int32_t)(h & 0x7fffu)) << 13;
    int32_t e = (int32_t)shifted_exp & o;
    o += (int32_t)(127 - 15) << 23;
    int32_t infnan = o + ((int32_t)(128 - 16) << 23);
    int32_t zeroden = (int32_t)f2u(u2f((uint32_t)o + (1u << 23)) - u2f(113u << 23));
    int32_t reg = (e == 0) ? zeroden : o;
    int32_t sign = ((int32_t)(h & 0x8000u)) << 16;
    return u2f((uint32_t)(((e == (int32_t)shifted_exp) ? infnan : reg) | sign));
}

uint16_t orc_float_to_half(float input) { /* float16.h:62-117 */
    uint32_t sign_mask = 0x80000000u;
    int32_t o;
    uint32_t fint = f2u(input);
    uint32_t sign = fint & sign_mask;
    fint ^= sign;
    uint32_t f32infty = 255u << 23;
    o = (fint > f32infty) ? 0x7e00 : 0x7c00;
    const uint32_t round_mask = ~0xfffu;
    const uint32_t magic = 15u << 23;
    float fscale = u2f(fint & round_mask) * u2f(magic);
    float cap = u2f((31u << 23) - 0x1000u);
    fscale = (cap < fscale) ? cap : fscale; /* std::min */
    int32_t fint2 = (int32_t)(f2u(fscale) - round_mask);
    if (fint < f32infty) o = fint2 >> 13;
    return (uint16_t)((uint32_t)o | (sign >> 16));
}

uint16_t orc_float_to_bf16(float ff) { /* bfloat16.h:22-29 */
    uint32_t f32 = f2u(ff);
    uint32_t lsb = (f32 >> 16) & 1;
    f32 += lsb + 0x7FFF;
    return (uint16_t)(f32 >> 16);
}
static inline float bf16_to_float(uint16_t b) { return u2f((uint32_t)b << 16); }

/* ------------------------------------------------------------------ distances -------------- */
/* fp32, scalar baseline: res += t*t with separate roundings (the TU is built without FMA). */
static float f32_l2_scalar(const float *a, const float *b, size_t d) {
    volatile float res = 0;
    for (size_t i = 0; i < d; i++) {
        volatile float t = a[i] - b[i];
        volatile float sq = t * t;
        res = res + sq;
    }
    return res;
}
static float f32_ip_scalar(const float *a, const float *b, size_t d) {
    volatile float res = 0;
    for (size_t i = 0; i < d; i++) {
        volatile float p = a[i] * b[i];
        res = res + p;
    }
    return 1.0f - res;
}

/* fp32, AVX-512F tier emulated: 2 x 16 accumulators, masked head multiply, odd 16-step into sum1,
 * pairs of steps into sum0/sum1, sum0+sum1, then the _mm512_reduce_add_ps tree
 * (halves of 8, 4, 2, 1). */
static float reduce16(const float *s) {
    float t8[8], t4[4], t2[2];
    for (int j = 0; j < 8; j++) t8[j] = s[j] + s[j + 8];
    for (int j = 0; j < 4; j++) t4[j] = t8[j] + t8[j + 4];
    for (int j = 0; j < 2; j++) t2[j] = t4[j] + t4[j + 2];
    return t2[0] + t2[1];
}
static float f32_avx512(const float *a, const float *b, size_t dim, int l2) {
    float s0[16], s1[16], s[16];
    for (int j = 0; j < 16; j++) s0[j] = s1[j] = 0.0f;
    const size_t residual = dim % 32, r16 = residual % 16;
    size_t p = 0;
    for (size_t j = 0; j < r16; j++) { /* masked multiply into sum0 */
        if (l2) {
            volatile float df = a[j] - b[j];
            volatile float m = df * df;
            s0[j] = m;
        } else {
            volatile float m = a[j] * b[j];
            s0[j] = m;
        }
    }
    p = r16;
    if (residual >= 16) {
        for (int j = 0; j < 16; j++) {
            if (l2) {
                volatile float df = a[p + j] - b[p + j];
                s1[j] = fmaf(df, df, s1[j]);
            } else {
                s1[j] = fmaf(a[p + j], b[p + j], s1[j]);
            }
        }
        p += 16;
    }
    while (p < dim) {
        for (int j = 0; j < 16; j++) {
            if (l2) {
                volatile float df = a[p + j] - b[p + j];
                s0[j] = fmaf(df, df, s0[j]);
            } else {
                s0[j] = fmaf(a[p + j], b[p + j], s0[j]);
            }
        }
        p += 16;
        for (int j = 0; j < 16; j++) {
            if (l2) {
                volatile float df = a[p + j] - b[p + j];
                s1[j] = fmaf(df, df, s1[j]);
            } else {
                s1[j] = fmaf(a[p + j], b[p + j], s1[j]);
            }
        }
        p += 16;
    }
    for (int j = 0; j < 16; j++) s[j] = s0[j] + s1[j];
    const float r = reduce16(s);
    return l2 ? r : 1.0f - r;
}

static float f16_dist(const uint16_t *a, const uint16_t *b, size_t d, int l2) { /* L2.cpp:123-132, IP.cpp:229-238 */
    volatile float res = 0;
    for (size_t i = 0; i < d; i++) {
        float x = orc_half_to_float(a[i]), y = orc_half_to_float(b[i]);
        if (l2) {
            volatile float t = x - y;
            volatile float sq = t * t;
            res = res + sq;
        } else {
            volatile float pr = x * y;
            res = res + pr;
        }
    }
    return l2 ? res : 1.0f - res;
}
static float bf16_dist(const uint16_t *a, const uint16_t *b, size_t d, int l2) { /* L2.cpp:100-121, IP.cpp:207-227 */
    volatile float res = 0;
    for (size_t i = 0; i < d; i++) {
        float x = bf16_to_float(a[i]), y = bf16_to_float(b[i]);
        if (l2) {
            volatile float t = x - y;
            volatile float sq = t * t;
            res = res + sq;
        } else {
            volatile float pr = x * y;
            res = res + pr;
        }
    }
    return l2 ? res : 1.0f - res;
}

static float int_dist(const uint8_t *a, const uint8_t *b, size_t d, int metric, int is_signed) {
    int acc = 0; /* ret_t<int8_t> == int: IP.cpp:243-252, L2.cpp:134-160 */
    for (size_t i = 0; i < d; i++) {
        int x = is_signed ? (int)(int8_t)a[i] : (int)a[i];
        int y = is_signed ? (int)(int8_t)b[i] : (int)b[i];
        if (metric == ORC_L2) {
            int16_t df = (int16_t)(x - y);
            acc += df * df;
        } else {
            acc += x * y;
        }
    }
    if (metric == ORC_L2) return (float)acc;
    if (metric == ORC_IP) return (float)(1 - acc);
    float n1, n2; /* IP.cpp:264-271: norms stored after the dim payload bytes */
    memcpy(&n1, a + d, 4);
    memcpy(&n2, b + d, 4);
    volatile float prod = n1 * n2;
    volatile float q = (float)acc / prod;
    return 1.0f - q;
}

float orc_distance(int type, int metric, size_t dim, const void *a, const void *b, int tier) {
    const int l2 = (metric == ORC_L2);
    switch (type) {
    case ORC_F32:
        if (tier == ORC_TIER_AVX512 && dim >= 8) return f32_avx512((const float *)a, (const float *)b, dim, l2);
        return l2 ? f32_l2_scalar((const float *)a, (const float *)b, dim) : f32_ip_scalar((const float *)a, (const float *)b, dim);
    case ORC_F16: return f16_dist((const uint16_t *)a, (const uint16_t *)b, dim, l2);
    case ORC_BF16: return bf16_dist((const uint16_t *)a, (const uint16_t *)b, dim, l2);
    case ORC_I8: return int_dist((const uint8_t *)a, (const uint8_t *)b, dim, metric, 1);
    case ORC_U8: return int_dist((const uint8_t *)a, (const uint8_t *)b, dim, metric, 0);
    }
    return NAN;
}

/* ------------------------------------------------------------------ normalisers ------------ */
void orc_normalize(void *blob, size_t dim, int type) {
    if (type == ORC_F32) { /* normalize_naive.h:23-37 */
        float *v = (float *)blob;
        double sum = 0;
        for (size_t i = 0; i < dim; i++) sum += (double)v[i] * (double)v[i];
        float norm = (float)sqrt(sum);
        for (size_t i = 0; i < dim; i++) v[i] = v[i] / norm;
    } else if (type == ORC_F16 || type == ORC_BF16) { /* :39-77 */
        uint16_t *v = (uint16_t *)blob;
        float *tmp = (float *)malloc(dim * sizeof(float));
        volatile float sum = 0;
        for (size_t i = 0; i < dim; i++) {
            float val = (type == ORC_F16) ? orc_half_to_float(v[i]) : bf16_to_float(v[i]);
            tmp[i] = val;
            volatile float sq = val * val;
            sum = sum + sq;
        }
        float norm = (float)sqrt((double)sum);
        for (size_t i = 0; i < dim; i++) {
            float q = tmp[i] / norm;
            v[i] = (type == ORC_F16) ? orc_float_to_half(q) : orc_float_to_bf16(q);
        }
        free(tmp);
    } else { /* :79-88 + compute_norm.h:17-28 */
        uint8_t *v = (uint8_t *)blob;
        int sum = 0;
        for (size_t i = 0; i < dim; i++) {
            int x = (type == ORC_I8) ? (int)(int8_t)v[i] : (int)v[i];
            sum += x * x;
        }
        float norm = (float)sqrt((double)sum);
        memcpy(v + dim, &norm, 4);
    }
}

size_t orc_stored_size(int type, size_t dim, int metric) {
    size_t es = (type == ORC_F32) ? 4 : (type == ORC_F16 || type == ORC_BF16) ? 2 : 1;
    size_t s = es * dim;
    if (metric == ORC_COS && (type == ORC_I8 || type == ORC_U8)) s += 4;
    return s;
}

/* ------------------------------------------------------------------ index ------------------- */
typedef struct {
    size_t label;
    uint32_t *ids;
    uint32_t n, cap;
    int used;
} LabelSlot;

struct OrcIndex {
    int type, metric, multi, tier;
    size_t dim, esize, row;  /* row = stored bytes */
    uint8_t *data;           /* count * row */
    size_t *id_to_label;
    size_t count, cap;
    LabelSlot *tab; /* open addressing label -> ids */
    size_t tab_cap, tab_used, n_labels;
};

static size_t hash_label(size_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}
static LabelSlot *tab_find(const OrcIndex *ix, size_t label, int create) {
    OrcIndex *m = (OrcIndex *)ix;
    if (m->tab_cap == 0 || (create && (m->tab_used + 1) * 2 > m->tab_cap)) {
        if (!create && m->tab_cap == 0) return NULL;
        size_t ncap = m->tab_cap ? m->tab_cap * 2 : 1024;
        LabelSlot *nt = (LabelSlot *)calloc(ncap, sizeof(LabelSlot));
        for (size_t i = 0; i < m->tab_cap; i++) {
            if (m->tab[i].used == 1) {
                size_t h = hash_label(m->tab[i].label) & (ncap - 1);
                while (nt[h].used) h = (h + 1) & (ncap - 1);
                nt[h] = m->tab[i];
            }
        }
        free(m->tab);
        m->tab = nt;
        m->tab_cap = ncap;
        size_t used = 0;
        for (size_t i = 0; i < ncap; i++) used += nt[i].used == 1;
        m->tab_used = used;
    }
    size_t h = hash_label(label) & (m->tab_cap - 1);
    LabelSlot *tomb = NULL;
    while (m->tab[h].used) {
        if (m->tab[h].used == 1 && m->tab[h].label == label) return &m->tab[h];
        if (m->tab[h].used == 2 && !tomb) tomb = &m->tab[h];
        h = (h + 1) & (m->tab_cap - 1);
    }
    if (!create) return NULL;
    LabelSlot *s = tomb ? tomb : &m->tab[h];
    if (!tomb) m->tab_used++;
    s->label = label;
    s->ids = NULL;
    s->n = s->cap = 0;
    s->used = 1;
    m->n_labels++;
    return s;
}
static void slot_push(LabelSlot *s, uint32_t id) {
    if (s->n == s->cap) {
        s->cap = s->cap ? s->cap * 2 : 1;
        s->ids = (uint32_t *)realloc(s->ids, s->cap * sizeof(uint32_t));
    }
    s->ids[s->n++] = id;
}

OrcIndex *orc_index_new(int type, size_t dim, int metric, int multi, int tier) {
    OrcIndex *ix = (OrcIndex *)calloc(1, sizeof(OrcIndex));
    ix->type = type;
    ix->metric = metric;
    ix->multi = multi;
    ix->tier = tier;
    ix->dim = dim;
    ix->esize = (type == ORC_F32) ? 4 : (type == ORC_F16 || type == ORC_BF16) ? 2 : 1;
    ix->row = orc_stored_size(type, dim, metric);
    return ix;
}
void orc_index_free(OrcIndex *ix) {
    if (!ix) return;
    for (size_t i = 0; i < ix->tab_cap; i++)
        if (ix->tab[i].used == 1) free(ix->tab[i].ids);
    free(ix->tab);
    free(ix->data);
    free(ix->id_to_label);
    free(ix);
}
size_t orc_index_size(const OrcIndex *ix) { return ix->count; }

static void preprocess(const OrcIndex *ix, const void *blob, uint8_t *dst) { /* preprocessors.h:49-146 */
    memcpy(dst, blob, ix->dim * ix->esize);
    if (ix->metric == ORC_COS) orc_normalize(dst, ix->dim, ix->type);
}

int orc_index_add(OrcIndex *ix, const void *blob, size_t label) {
    if (!ix->multi) {
        LabelSlot *s = tab_find(ix, label, 0);
        if (s) { /* brute_force_single.h:139-144: raw blob overwrites the stored row */
            uint8_t *dst = ix->data + (size_t)s->ids[0] * ix->row;
            memcpy(dst, blob, ix->dim * ix->esize);
            if (ix->metric == ORC_COS && (ix->type == ORC_I8 || ix->type == ORC_U8)) orc_normalize(dst, ix->dim, ix->type);
            return 0;
        }
    }
    if (ix->count == ix->cap) {
        ix->cap = ix->cap ? ix->cap * 2 : 1024;
        ix->data = (uint8_t *)realloc(ix->data, ix->cap * ix->row);
        ix->id_to_label = (size_t *)realloc(ix->id_to_label, ix->cap * sizeof(size_t));
    }
    preprocess(ix, blob, ix->data + ix->count * ix->row);
    ix->id_to_label[ix->count] = label;
    slot_push(tab_find(ix, label, 1), (uint32_t)ix->count);
    ix->count++;
    return 1;
}
void orc_index_add_bulk(OrcIndex *ix, const void *blobs, size_t stride, size_t n, size_t label0) {
    for (size_t i = 0; i < n; i++) orc_index_add(ix, (const uint8_t *)blobs + i * stride, label0 + i);
}

static void remove_id(OrcIndex *ix, uint32_t id) { /* brute_force.h:196-224 */
    uint32_t last = (uint32_t)(--ix->count);
    if (id != last) {
        size_t last_label = ix->id_to_label[last];
        ix->id_to_label[id] = last_label;
        LabelSlot *s = tab_find(ix, last_label, 0);
        for (uint32_t i = 0; i < s->n; i++)
            if (s->ids[i] == last) s->ids[i] = id;
        memcpy(ix->data + (size_t)id * ix->row, ix->data + (size_t)last * ix->row, ix->row);
    }
}
int orc_index_delete(OrcIndex *ix, size_t label) {
    LabelSlot *s = tab_find(ix, label, 0);
    if (!s) return 0;
    uint32_t n = s->n;
    uint32_t *ids = s->ids;
    s->used = 2;
    s->ids = NULL;
    ix->n_labels--;
    /* delete highest ids first so that earlier swaps never move another victim */
    for (uint32_t i = 0; i < n; i++)
        for (uint32_t j = i + 1; j < n; j++)
            if (ids[j] > ids[i]) {
                uint32_t t = ids[i];
                ids[i] = ids[j];
                ids[j] = t;
            }
    for (uint32_t i = 0; i < n; i++) remove_id(ix, ids[i]);
    free(ids);
    return (int)n;
}

/* pair<float,size_t> ordering of the reference heap */
typedef struct {
    float score;
    size_t label;
} Pair;
static int pair_less(Pair a, Pair b) { return a.score < b.score || (!(b.score < a.score) && a.label < b.label); }

static void heap_push(Pair *h, size_t *n, Pair v) {
    size_t i = (*n)++;
    h[i] = v;
    while (i) {
        size_t p = (i - 1) / 2;
        if (!pair_less(h[p], h[i])) break;
        Pair t = h[p];
        h[p] = h[i];
        h[i] = t;
        i = p;
    }
}
static void heap_pop(Pair *h, size_t *n) {
    h[0] = h[--(*n)];
    size_t i = 0;
    for (;;) {
        size_t l = 2 * i + 1, r = l + 1, m = i;
        if (l < *n && pair_less(h[m], h[l])) m = l;
        if (r < *n && pair_less(h[m], h[r])) m = r;
        if (m == i) break;
        Pair t = h[m];
        h[m] = h[i];
        h[i] = t;
        i = m;
    }
}

static int cmp_pair_score(const void *a, const void *b) {
    const Pair *x = (const Pair *)a, *y = (const Pair *)b;
    if (pair_less(*x, *y)) return -1;
    if (pair_less(*y, *x)) return 1;
    return 0;
}
static int cmp_pair_label(const void *a, const void *b) {
    const Pair *x = (const Pair *)a, *y = (const Pair *)b;
    return (x->label > y->label) - (x->label < y->label);
}

static float dist_row(const OrcIndex *ix, size_t id, const void *q) {
    return orc_distance(ix->type, ix->metric, ix->dim, ix->data + id * ix->row, q, ix->tier);
}

size_t orc_index_topk(const OrcIndex *ix, const void *query, size_t k, int order, size_t *labels, double *scores) {
    if (k == 0 || ix->count == 0) return 0; /* brute_force.h:251-253 */
    uint8_t *q = (uint8_t *)malloc(ix->row + 16);
    preprocess(ix, query, q);
    size_t n = 0;
    Pair *out = NULL;
    if (!ix->multi) {
        Pair *heap = (Pair *)malloc((k + 1) * sizeof(Pair));
        float upper = -INFINITY; /* numeric_limits<float>::lowest() is finite, but nothing is below it */
        upper = -3.402823466e+38F;
        for (size_t id = 0; id < ix->count; id++) { /* :264-281 */
            float s = dist_row(ix, id, q);
            if (s < upper || n < k) {
                Pair p = {s, ix->id_to_label[id]};
                heap_push(heap, &n, p);
                if (n > k) heap_pop(heap, &n);
                upper = heap[0].score;
            }
        }
        out = heap;
    } else {
        /* updatable_max_heap semantics (VS/utils/updatable_heap.h:25-113): best score per label,
         * then the k best labels. */
        Pair *best = (Pair *)malloc(ix->n_labels * sizeof(Pair));
        size_t nb = 0;
        for (size_t i = 0; i < ix->tab_cap; i++) {
            if (ix->tab[i].used != 1) continue;
            Pair p = {INFINITY, ix->tab[i].label};
            int first = 1;
            for (uint32_t j = 0; j < ix->tab[i].n; j++) {
                float s = dist_row(ix, ix->tab[i].ids[j], q);
                if (first || s < p.score) p.score = s;
                first = 0;
            }
            best[nb++] = p;
        }
        qsort(best, nb, sizeof(Pair), cmp_pair_score);
        n = nb < k ? nb : k;
        out = best;
    }
    qsort(out, n, sizeof(Pair), order == 1 ? cmp_pair_label : cmp_pair_score);
    for (size_t i = 0; i < n; i++) {
        labels[i] = out[i].label;
        scores[i] = (double)out[i].score;
    }
    free(out);
    free(q);
    return n;
}

size_t orc_index_range(const OrcIndex *ix, const void *query, double radius, int order, size_t cap, size_t *labels,
                       double *scores) {
    uint8_t *q = (uint8_t *)malloc(ix->row + 16);
    preprocess(ix, query, q);
    const float r = (float)radius;
    Pair *res = (Pair *)malloc((ix->count + 1) * sizeof(Pair));
    size_t n = 0;
    if (!ix->multi) {
        for (size_t id = 0; id < ix->count; id++) {
            float s = dist_row(ix, id, q);
            if (s <= r) {
                res[n].score = s;
                res[n++].label = ix->id_to_label[id];
            }
        }
    } else {
        for (size_t i = 0; i < ix->tab_cap; i++) {
            if (ix->tab[i].used != 1) continue;
            int any = 0;
            float bs = 0;
            for (uint32_t j = 0; j < ix->tab[i].n; j++) {
                float s = dist_row(ix, ix->tab[i].ids[j], q);
                if (s <= r && (!any || s < bs)) {
                    bs = s;
                    any = 1;
                }
            }
            if (any) {
                res[n].score = bs;
                res[n++].label = ix->tab[i].label;
            }
        }
    }
    qsort(res, n, sizeof(Pair), order == 1 ? cmp_pair_label : cmp_pair_score);
    for (size_t i = 0; i < n && i < cap; i++) {
        labels[i] = res[i].label;
        scores[i] = (double)res[i].score;
    }
    free(res);
    free(q);
    return n;
}

double orc_index_distance_from(const OrcIndex *ix, size_t label, const void *stored_form_query) {
    LabelSlot *s = tab_find(ix, label, 0);
    if (!s) return NAN; /* brute_force_single.h:204-207 */
    /* brute_force_multi.h:234-238: `dist = (dist < d) ? dist : d` from +inf in the label's row order, so a NaN row replaces
     * the running value and the next row replaces the NaN: NaN exactly when the last row is NaN */
    float best = INFINITY;
    for (uint32_t j = 0; j < s->n; j++) {
        const float d = dist_row(ix, s->ids[j], stored_form_query);
        best = (best < d) ? best : d;
    }
    return (double)best;
}

int orc_index_prefer_adhoc(const OrcIndex *ix, size_t subset, size_t k, int initial) {
    (void)k;
    (void)initial;
    size_t index_size = ix->count;
    if (subset > index_size) subset = index_size;
    size_t d = ix->dim;
    float r = (index_size == 0) ? 0.0f : (float)subset / (float)ix->n_labels;
    if (index_size <= 5500) return 1;
    if (d <= 300) {
        if (r <= 0.15) return 1;
        if (r <= 0.35) {
            if (d <= 75) return 0;
            return index_size <= 550000;
        }
        return 0;
    }
    if (r <= 0.55) return 1;
    if (d <= 750) return 0;
    return r <= 0.75;
}

size_t orc_index_all_sorted(const OrcIndex *ix, const void *query, size_t *labels, double *scores) {
    return orc_index_topk(ix, query, ix->count ? ix->count : 1, 0, labels, scores);
}

/* ------------------------------------------------------------------ timing ------------------ */
typedef struct {
    const OrcIndex *ix;
    const uint8_t *queries;
    size_t qstride, nq, k;
    size_t *labels;
    double *scores;
    size_t *next;
    pthread_mutex_t *mu;
} Work;
static void *worker(void *arg) {
    Work *w = (Work *)arg;
    size_t *l = (size_t *)malloc(w->k * sizeof(size_t));
    double *s = (double *)malloc(w->k * sizeof(double));
    for (;;) {
        pthread_mutex_lock(w->mu);
        size_t i = (*w->next)++;
        pthread_mutex_unlock(w->mu);
        if (i >= w->nq) break;
        size_t n = orc_index_topk(w->ix, w->queries + i * w->qstride, w->k, 0, l, s);
        for (size_t j = 0; j < n; j++) {
            if (w->labels) w->labels[i * w->k + j] = l[j];
            if (w->scores) w->scores[i * w->k + j] = s[j];
        }
    }
    free(l);
    free(s);
    return NULL;
}
double orc_index_time_topk(const OrcIndex *ix, const void *queries, size_t qstride, size_t nq, size_t k, int nthreads,
                           size_t *labels, double *scores) {
    pthread_mutex_t mu = PTHREAD_MUTEX_INITIALIZER;
    size_t next = 0;
    Work w = {ix, (const uint8_t *)queries, qstride, nq, k, labels, scores, &next, &mu};
    if (nthreads < 1) nthreads = 1;
    pthread_t *th = (pthread_t *)malloc((size_t)nthreads * sizeof(pthread_t));
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int t = 0; t < nthreads; t++) pthread_create(&th[t], NULL, worker, &w);
    for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    clock_gettime(CLOCK_MONOTONIC, &t1);
    free(th);
    return (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
}

/* Streaming form of orc_index_topk over a flat array of stored-form rows handed over chunk by chunk (the fallback of
 * oracle/ref_shim/ref_capi.cpp Ref_ScanTopKChunk when oracle/_ref is not built): brute_force.h:262-281 admission rule on
 * the same heap, state carried in labels/scores/counts between chunks, labels = label0 + row index. */
typedef struct {
    int type, metric, tier;
    size_t dim, stride, n, label0, qstride, nq, k;
    const uint8_t *rows, *queries;
    size_t *labels, *counts;
    float *scores;
    size_t *next;
    pthread_mutex_t *mu;
} ScanWork;
static void *scan_worker(void *arg) {
    ScanWork *w = (ScanWork *)arg;
    Pair *heap = (Pair *)malloc((w->k + 1) * sizeof(Pair));
    for (;;) {
        pthread_mutex_lock(w->mu);
        size_t qi = (*w->next)++;
        pthread_mutex_unlock(w->mu);
        if (qi >= w->nq) break;
        const void *q = w->queries + qi * w->qstride;
        size_t hn = 0;
        for (size_t j = 0; j < w->counts[qi]; j++) {
            Pair v = {w->scores[qi * w->k + j], w->labels[qi * w->k + j]};
            heap_push(heap, &hn, v);
        }
        float upper = hn ? heap[0].score : -FLT_MAX;
        for (size_t r = 0; r < w->n; r++) {
            float sc = orc_distance(w->type, w->metric, w->dim, w->rows + r * w->stride, q, w->tier);
            if (sc < upper || hn < w->k) {
                Pair v = {sc, w->label0 + r};
                heap_push(heap, &hn, v);
                if (hn > w->k) heap_pop(heap, &hn);
                upper = heap[0].score;
            }
        }
        size_t c = 0;
        while (hn) {
            w->scores[qi * w->k + c] = heap[0].score;
            w->labels[qi * w->k + c] = heap[0].label;
            heap_pop(heap, &hn);
            c++;
        }
        w->counts[qi] = c;
    }
    free(heap);
    return NULL;
}
void orc_scan_topk_chunk(int type, int metric, int tier, size_t dim, const void *rows, size_t stride, size_t n, size_t label0,
                         const void *queries, size_t qstride, size_t nq, size_t k, int nthreads, size_t *labels, float *scores,
                         size_t *counts) {
    pthread_mutex_t mu = PTHREAD_MUTEX_INITIALIZER;
    size_t next = 0;
    ScanWork w = {type, metric, tier, dim, stride, n, label0, qstride, nq, k, (const uint8_t *)rows, (const uint8_t *)queries,
                  labels, counts, scores, &next, &mu};
    if (nthreads < 1) nthreads = 1;
    pthread_t *th = (pthread_t *)malloc((size_t)nthreads * sizeof(pthread_t));
    for (int t = 0; t < nthreads; t++) pthread_create(&th[t], NULL, scan_worker, &w);
    for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    free(th);
}

/* ------------------------------------------------------------------ synthetic data ---------- */
uint64_t orc_mix64(uint64_t seed, uint64_t a, uint64_t b) { /* splitmix64-style finaliser chain */
    uint64_t z = seed + 0x9E3779B97F4A7C15ULL * (a + 1) + 0xD1B54A32D192ED03ULL * (b + 1);
    z ^= z >> 30;
    z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27;
    z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
float orc_synth_f32(uint64_t seed, uint64_t row, uint64_t col) {
    uint32_t m = (uint32_t)(orc_mix64(seed, row, col) >> 40); /* 24 random bits */
    return (float)m * (2.0f / 16777216.0f) - 1.0f;            /* exact in fp32 */
}
void orc_synth_rows(int type, uint64_t seed, uint64_t row0, size_t nrows, size_t dim, void *out) {
    for (size_t r = 0; r < nrows; r++)
        for (size_t c = 0; c < dim; c++) {
            float x = orc_synth_f32(seed, row0 + r, c);
            size_t i = r * dim + c;
            switch (type) {
            case ORC_F32: ((float *)out)[i] = x; break;
            case ORC_F16: ((uint16_t *)out)[i] = orc_float_to_half(x); break;
            case ORC_BF16: ((uint16_t *)out)[i] = orc_float_to_bf16(x); break;
            case ORC_I8: ((int8_t *)out)[i] = (int8_t)lrintf(127.0f * x); break;
            case ORC_U8: ((uint8_t *)out)[i] = (uint8_t)lrintf(127.5f * x + 127.5f); break;
            }
        }
}
