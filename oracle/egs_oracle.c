/*
 * egs_oracle.c -- CPU ORACLE: TEST INFRASTRUCTURE ONLY (see egs_oracle.h).
 *
 * Plain-C restatement of pkg/scheduler of elastic-ai/elastic-gpu-scheduler;
 * each function cites the reference file:line it follows.  All arithmetic is
 * int64_t because Go's `int` is 64-bit on the reference's platforms.
 * "parity unpinned" by the reference's own tests; pinned by SURVEY.md 8c vectors.
 */
#define _GNU_SOURCE
#include "egs_oracle.h"

#include <pthread.h>
#include <sched.h>
#include <stdatomic.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define CORE_EACH_CARD 100 /* pkg/utils/types.go:6 */
#define NOT_NEED_GPU (-1)  /* allocate.go:16 */
#define NOT_NEED_RATE (-2) /* allocate.go:17 */

enum { ST_OK = 0, ST_NOFIT = 1, ST_NO_OPTION = 2, ST_TRANSACT = 3, ST_BAD_ARG = 4, ST_PANIC = 9 };

/* ---------------------------------------------------------------- sha256 (FIPS 180-4) */
static const uint32_t K256[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5,
    0xd807aa98, 0x12835b01, 0x243185be, 0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174,
    0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa, 0x5cb0a9dc, 0x76f988da,
    0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967,
    0x27b70a85, 0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85,
    0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3, 0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070,
    0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f, 0x682e6ff3,
    0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
#define ROR(x, n) (((x) >> (n)) | ((x) << (32 - (n))))
static void sha256_block(uint32_t h[8], const uint8_t *p) {
  uint32_t w[64];
  for (int i = 0; i < 16; i++)
    w[i] = (uint32_t)p[4 * i] << 24 | (uint32_t)p[4 * i + 1] << 16 | (uint32_t)p[4 * i + 2] << 8 | p[4 * i + 3];
  for (int i = 16; i < 64; i++) {
    uint32_t s0 = ROR(w[i - 15], 7) ^ ROR(w[i - 15], 18) ^ (w[i - 15] >> 3);
    uint32_t s1 = ROR(w[i - 2], 17) ^ ROR(w[i - 2], 19) ^ (w[i - 2] >> 10);
    w[i] = w[i - 16] + s0 + w[i - 7] + s1;
  }
  uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
  for (int i = 0; i < 64; i++) {
    uint32_t S1 = ROR(e, 6) ^ ROR(e, 11) ^ ROR(e, 25);
    uint32_t ch = (e & f) ^ (~e & g);
    uint32_t t1 = hh + S1 + ch + K256[i] + w[i];
    uint32_t S0 = ROR(a, 2) ^ ROR(a, 13) ^ ROR(a, 22);
    uint32_t mj = (a & b) ^ (a & c) ^ (b & c);
    uint32_t t2 = S0 + mj;
    hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
  }
  h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
}
void egso_sha256(const uint8_t *msg, uint64_t len, uint8_t out[32]) {
  uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
  uint64_t i = 0;
  for (; i + 64 <= len; i += 64) sha256_block(h, msg + i);
  uint8_t tail[128];
  uint64_t r = len - i;
  memcpy(tail, msg + i, r);
  tail[r++] = 0x80;
  uint64_t padded = (r <= 56) ? 64 : 128;
  memset(tail + r, 0, padded - r);
  uint64_t bits = len * 8;
  for (int k = 0; k < 8; k++) tail[padded - 1 - k] = (uint8_t)(bits >> (8 * k));
  sha256_block(h, tail);
  if (padded == 128) sha256_block(h, tail + 64);
  for (int k = 0; k < 8; k++) {
    out[4 * k] = h[k] >> 24; out[4 * k + 1] = h[k] >> 16; out[4 * k + 2] = h[k] >> 8; out[4 * k + 3] = h[k];
  }
}

/* GPUUnit.String gpu.go:15-17 + GPURequest.String allocate.go:22-28 */
static int request_string(int C, const egso_unit *u, char *buf, size_t cap) {
  int n = 0;
  for (int i = 0; i < C; i++)
    n += snprintf(buf + n, cap - n, "(core: %lld, memory: %lld, gpu count: %lld)", (long long)u[i].core,
                  (long long)u[i].mem, (long long)u[i].count);
  return n;
}
/* GPURequest.Hash allocate.go:30-33: first 8 hex chars == first 4 digest bytes */
static uint32_t request_key32(int C, const egso_unit *u) {
  char buf[EGSO_MAX_C * 96];
  int n = request_string(C, u, buf, sizeof buf);
  uint8_t d[32];
  egso_sha256((const uint8_t *)buf, (uint64_t)n, d);
  return (uint32_t)d[0] << 24 | (uint32_t)d[1] << 16 | (uint32_t)d[2] << 8 | d[3];
}
void egso_request_hash(int C, const egso_unit *units, char out[9]) {
  snprintf(out, 9, "%08x", request_key32(C, units));
}
/* NewGPURequest, allocate.go:38-53 */
void egso_unit_from_requests(int64_t core, int64_t mem, egso_unit *out) {
  out->core = out->mem = out->count = 0;
  if (core == 0 && mem == 0) { out->core = NOT_NEED_GPU; out->mem = NOT_NEED_GPU; return; }
  if (core >= CORE_EACH_CARD) { out->count = core / CORE_EACH_CARD; return; }
  out->core = core; out->mem = mem;
}

uint64_t egso_mix64(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

/* ---------------------------------------------------------------- data model */
typedef struct { int64_t ca, ma, ct, mt; } gpu_t; /* GPU, gpu.go:19-25 */

typedef struct {          /* GPUOption, allocate.go:60-73 */
  uint32_t key;           /* shape id, or sha256 prefix when faithful */
  int C;
  int64_t score;
  int8_t n[EGSO_MAX_C];
  int8_t idx[EGSO_MAX_C][EGSO_MAX_G];
} opt_t;

typedef struct {          /* NodeAllocator, node.go:13-21 */
  int G;
  gpu_t g[EGSO_MAX_G];
  opt_t *cache; int nc, cc;          /* allocated map[string]*GPUOption */
  uint64_t *pods; int np, pc;        /* podsMap */
} node_t;

typedef struct { uint64_t *k; uint8_t *s; size_t cap, used; } u64set; /* s: 0 empty 1 full 2 tomb */

typedef struct { int C; egso_unit u[EGSO_MAX_C]; } shape_t;

struct pool;
struct egso {
  int policy, faithful;
  node_t *nodes; int nn, nc;
  shape_t *shapes; int ns, sc;
  u64set pod_maps, released;        /* BaseScheduler.podMaps / releasedPodMap, scheduler.go:47-49 */
  struct pool *pool;
};

static void set_init(u64set *s) { s->cap = 0; s->used = 0; s->k = NULL; s->s = NULL; }
static void set_free(u64set *s) { free(s->k); free(s->s); }
static size_t set_slot(const u64set *s, uint64_t key, int *found) {
  size_t m = s->cap - 1, i = (size_t)egso_mix64(key) & m, tomb = (size_t)-1;
  for (;;) {
    if (s->s[i] == 0) { *found = 0; return tomb != (size_t)-1 ? tomb : i; }
    if (s->s[i] == 1 && s->k[i] == key) { *found = 1; return i; }
    if (s->s[i] == 2 && tomb == (size_t)-1) tomb = i;
    i = (i + 1) & m;
  }
}
static int set_has(const u64set *s, uint64_t key) {
  if (!s->cap) return 0;
  int f; set_slot(s, key, &f); return f;
}
static void set_add(u64set *s, uint64_t key);
static void set_grow(u64set *s) {
  u64set o = *s;
  s->cap = o.cap ? o.cap * 2 : 1024; s->used = 0;
  s->k = calloc(s->cap, sizeof *s->k); s->s = calloc(s->cap, 1);
  for (size_t i = 0; i < o.cap; i++) if (o.s[i] == 1) set_add(s, o.k[i]);
  free(o.k); free(o.s);
}
static void set_add(u64set *s, uint64_t key) {
  if ((s->used + 1) * 2 > s->cap) set_grow(s);
  int f; size_t i = set_slot(s, key, &f);
  if (f) return;
  if (s->s[i] == 0) s->used++;
  s->s[i] = 1; s->k[i] = key;
}
static void set_del(u64set *s, uint64_t key) {
  if (!s->cap) return;
  int f; size_t i = set_slot(s, key, &f);
  if (f) s->s[i] = 2;
}

/* ---------------------------------------------------------------- GPU arithmetic */
static inline void gpu_add(gpu_t *g, const egso_unit *u) { /* gpu.go:31-39 */
  if (u->count > 0) { g->ca = 0; g->ma = 0; } else { g->ca -= u->core; g->ma -= u->mem; }
}
static inline void gpu_sub(gpu_t *g, const egso_unit *u) { /* gpu.go:41-49 */
  if (u->count > 0) { g->ca = g->ct; g->ma = g->mt; } else { g->ca += u->core; g->ma += u->mem; }
}
static inline int gpu_can(const gpu_t *g, const egso_unit *u) { /* gpu.go:51-56 */
  if (u->count > 0) return g->ca == g->ct && g->ma == g->mt;
  return g->ca >= u->core && g->ma >= u->mem;
}

/* Binpack.Rate rater.go:18-51 / Spread.Rate rater.go:56-59 */
static int64_t rate(int policy, const gpu_t *g, int G, const int *idx, int C) {
  if (policy != 0) return 0;
  int seen[EGSO_MAX_G] = {0}, k = 0;
  for (int i = 0; i < C; i++) {
    if (idx[i] < 0) continue;
    if (!seen[idx[i]]) { seen[idx[i]] = 1; k++; }
  }
  int64_t maxm = g[0].ma, minm = g[0].ma, maxc = g[0].ca, minc = g[0].ca;
  for (int i = 0; i < G; i++) {
    if (g[i].ma > maxm) maxm = g[i].ma;
    if (g[i].ma < minm) minm = g[i].ma;
    if (g[i].ca > maxc) maxc = g[i].ca;
    if (g[i].ca < minc) minc = g[i].ca;
  }
  int64_t range = (maxm + maxc - minm - minc) / 2; /* C99 '/' truncates toward zero like Go */
  return range / (k + 1) * 100;
}

typedef struct {
  int policy, G, C, found;
  gpu_t *g;
  const egso_unit *req;
  int8_t n[EGSO_MAX_C];
  int8_t idx[EGSO_MAX_C][EGSO_MAX_G];
  opt_t best;
} trade_t;

/* the dfs closure of GPUs.Trade, gpu.go:72-123 */
static void trade_dfs(trade_t *t, int ci) {
  if (ci == t->C) { /* gpu.go:73-93 */
    t->found = 1;
    int ridx[EGSO_MAX_C];
    for (int i = 0; i < t->C; i++) ridx[i] = (t->n[i] == 1) ? t->idx[i][0] : NOT_NEED_RATE;
    int64_t s = rate(t->policy, t->g, t->G, ridx, t->C);
    if (t->best.score > s) return; /* gpu.go:85 */
    memcpy(t->best.n, t->n, sizeof t->n);
    memcpy(t->best.idx, t->idx, sizeof t->idx);
    t->best.score = s;
    return;
  }
  const egso_unit *u = &t->req[ci];
  if (u->count > 0) { /* gpu.go:95-109; GetFreeGPUs gpu.go:193-202 */
    int nf = 0; int8_t freeg[EGSO_MAX_G];
    for (int i = 0; i < t->G; i++)
      if (t->g[i].ca == t->g[i].ct && t->g[i].ma == t->g[i].mt) freeg[nf++] = (int8_t)i;
    if (nf < u->count) return;
    t->n[ci] = (int8_t)u->count;
    for (int j = 0; j < u->count; j++) t->idx[ci][j] = freeg[j];
    for (int j = 0; j < u->count; j++) gpu_add(&t->g[freeg[j]], u);
    trade_dfs(t, ci + 1);
    for (int j = 0; j < u->count; j++) gpu_sub(&t->g[freeg[j]], u);
    return;
  }
  for (int i = 0; i < t->G; i++) { /* gpu.go:110-122 */
    if (!gpu_can(&t->g[i], u)) continue;
    gpu_add(&t->g[i], u);
    t->n[ci] = 1; t->idx[ci][0] = (int8_t)i;
    trade_dfs(t, ci + 1);
    gpu_sub(&t->g[i], u);
  }
}

/* GPUs.Trade gpu.go:65-129; 1 = fit (option filled), 0 = "no enough resource to allocate" */
static int trade(int policy, node_t *nd, int C, const egso_unit *req, opt_t *out) {
  trade_t t;
  t.policy = policy; t.G = nd->G; t.C = C; t.found = 0; t.g = nd->g; t.req = req;
  memset(t.n, 0, sizeof t.n); memset(t.idx, 0, sizeof t.idx);
  memset(&t.best, 0, sizeof t.best);
  trade_dfs(&t, 0);
  if (!t.found) return 0;
  *out = t.best; out->C = C;
  return 1;
}

/* GPUs.Transact gpu.go:153-175: 1 ok, 0 error with earlier Adds kept */
static int transact(node_t *nd, int C, const egso_unit *req, const opt_t *o) {
  for (int i = 0; i < C; i++) {
    if (req[i].count > 0) {
      for (int j = 0; j < o->n[i]; j++) {
        gpu_t *g = &nd->g[o->idx[i][j]];
        if (!gpu_can(g, &req[i])) return 0;
        gpu_add(g, &req[i]);
      }
    } else if (o->n[i] > 0) {
      gpu_t *g = &nd->g[o->idx[i][0]];
      if (!gpu_can(g, &req[i])) return 0;
      gpu_add(g, &req[i]);
    }
  }
  return 1;
}
/* GPUs.Cancel gpu.go:177-191 */
static void cancel(node_t *nd, int C, const egso_unit *req, const opt_t *o) {
  for (int i = 0; i < C; i++) {
    if (req[i].count > 0) {
      for (int j = 0; j < o->n[i]; j++) gpu_sub(&nd->g[o->idx[i][j]], &req[i]);
    } else if (o->n[i] > 0) {
      gpu_sub(&nd->g[o->idx[i][0]], &req[i]);
    }
  }
}

/* ---------------------------------------------------------------- node level */
static opt_t *cache_find(node_t *nd, uint32_t key) {
  for (int i = 0; i < nd->nc; i++) if (nd->cache[i].key == key) return &nd->cache[i];
  return NULL;
}
static void cache_put(node_t *nd, const opt_t *o) {
  if (nd->nc == nd->cc) { nd->cc = nd->cc ? nd->cc * 2 : 4; nd->cache = realloc(nd->cache, nd->cc * sizeof(opt_t)); }
  nd->cache[nd->nc++] = *o;
}
static void cache_del(node_t *nd, uint32_t key) {
  for (int i = 0; i < nd->nc; i++) if (nd->cache[i].key == key) { nd->cache[i] = nd->cache[--nd->nc]; return; }
}
static int pods_has(node_t *nd, uint64_t uid) {
  for (int i = 0; i < nd->np; i++) if (nd->pods[i] == uid) return 1;
  return 0;
}
static void pods_add(node_t *nd, uint64_t uid) {
  if (nd->np == nd->pc) { nd->pc = nd->pc ? nd->pc * 2 : 4; nd->pods = realloc(nd->pods, nd->pc * sizeof(uint64_t)); }
  nd->pods[nd->np++] = uid;
}
static void pods_del(node_t *nd, uint64_t uid) {
  for (int i = 0; i < nd->np; i++) if (nd->pods[i] == uid) { nd->pods[i] = nd->pods[--nd->np]; return; }
}

static uint32_t intern(egso *o, int C, const egso_unit *u) {
  for (int i = 0; i < o->ns; i++)
    if (o->shapes[i].C == C && memcmp(o->shapes[i].u, u, C * sizeof *u) == 0) return (uint32_t)i;
  if (o->ns == o->sc) { o->sc = o->sc ? o->sc * 2 : 16; o->shapes = realloc(o->shapes, o->sc * sizeof(shape_t)); }
  o->shapes[o->ns].C = C;
  memset(o->shapes[o->ns].u, 0, sizeof o->shapes[o->ns].u);
  memcpy(o->shapes[o->ns].u, u, C * sizeof *u);
  return (uint32_t)o->ns++;
}
/* node.go:62-63 / :76-77 / :88-89: the reference rebuilds + hashes the request per node */
static inline uint32_t node_key(const egso *o, uint32_t shape, int C, const egso_unit *u) {
  return o->faithful ? request_key32(C, u) : shape;
}

/* NodeAllocator.Assume node.go:61-73 -> option or NULL */
static opt_t *node_assume(egso *o, node_t *nd, uint32_t shape, int C, const egso_unit *u) {
  uint32_t key = node_key(o, shape, C, u);
  opt_t *hit = cache_find(nd, key);
  if (hit) return hit;
  opt_t op;
  if (!trade(o->policy, nd, C, u, &op)) return NULL;
  op.key = key;
  cache_put(nd, &op);
  return &nd->cache[nd->nc - 1];
}

/* ---------------------------------------------------------------- worker pool (scheduler.go:129-156) */
typedef struct pool {
  int nthreads;
  pthread_t *th;
  atomic_int gen, done, next, stop;
  egso *o; int n; const int32_t *ids; uint32_t shape; int C; const egso_unit *u; uint8_t *fit;
} pool_t;

static void filter_range(egso *o, int lo, int hi, const int32_t *ids, uint32_t shape, int C,
                         const egso_unit *u, uint8_t *fit) {
  for (int i = lo; i < hi; i++) {
    int nid = ids ? ids[i] : i;
    if (nid < 0 || nid >= o->nn || o->nodes[nid].G == 0) { fit[i] = 0; continue; }
    fit[i] = node_assume(o, &o->nodes[nid], shape, C, u) != NULL;
  }
}
static void pool_work(pool_t *p) {
  for (;;) {
    int lo = atomic_fetch_add(&p->next, 64);
    if (lo >= p->n) break;
    int hi = lo + 64 < p->n ? lo + 64 : p->n;
    filter_range(p->o, lo, hi, p->ids, p->shape, p->C, p->u, p->fit);
  }
}
static void *pool_main(void *arg) {
  pool_t *p = arg;
  int seen = 0;
  for (;;) {
    int spins = 0;
    while (atomic_load_explicit(&p->gen, memory_order_acquire) == seen) {
      if (atomic_load(&p->stop)) return NULL;
      if (++spins > 2000) { sched_yield(); spins = 0; }
    }
    seen++;
    pool_work(p);
    atomic_fetch_add_explicit(&p->done, 1, memory_order_release);
  }
}
static pool_t *pool_get(egso *o, int threads) {
  if (o->pool && o->pool->nthreads == threads) return o->pool;
  if (o->pool) {
    atomic_store(&o->pool->stop, 1);
    for (int i = 0; i < o->pool->nthreads - 1; i++) pthread_join(o->pool->th[i], NULL);
    free(o->pool->th); free(o->pool); o->pool = NULL;
  }
  pool_t *p = calloc(1, sizeof *p);
  p->nthreads = threads; p->o = o;
  p->th = calloc(threads, sizeof(pthread_t));
  for (int i = 0; i < threads - 1; i++) pthread_create(&p->th[i], NULL, pool_main, p);
  o->pool = p;
  return p;
}

/* ---------------------------------------------------------------- public API */
egso *egso_create(int policy, int faithful) {
  egso *o = calloc(1, sizeof *o);
  o->policy = policy; o->faithful = faithful;
  set_init(&o->pod_maps); set_init(&o->released);
  return o;
}
void egso_destroy(egso *o) {
  if (!o) return;
  if (o->pool) {
    atomic_store(&o->pool->stop, 1);
    for (int i = 0; i < o->pool->nthreads - 1; i++) pthread_join(o->pool->th[i], NULL);
    free(o->pool->th); free(o->pool);
  }
  for (int i = 0; i < o->nn; i++) { free(o->nodes[i].cache); free(o->nodes[i].pods); }
  free(o->nodes); free(o->shapes); set_free(&o->pod_maps); set_free(&o->released); free(o);
}
/* NewNodeAllocator node.go:23-59 */
int egso_add_node(egso *o, int64_t core_allocatable, int64_t mem_allocatable) {
  if (o->nn == o->nc) { o->nc = o->nc ? o->nc * 2 : 64; o->nodes = realloc(o->nodes, o->nc * sizeof(node_t)); }
  node_t *nd = &o->nodes[o->nn++];
  memset(nd, 0, sizeof *nd);
  int64_t G = core_allocatable / CORE_EACH_CARD; /* node.go:27 */
  if (G == 0 || G > EGSO_MAX_G) return -1;       /* node.go:28-30 */
  nd->G = (int)G;
  int64_t m = mem_allocatable / G;               /* node.go:37-38 */
  for (int i = 0; i < nd->G; i++) { nd->g[i].ca = nd->g[i].ct = CORE_EACH_CARD; nd->g[i].ma = nd->g[i].mt = m; }
  return o->nn - 1;
}
int egso_num_nodes(egso *o) { return o->nn; }
int egso_gpu_count(egso *o, int node) { return o->nodes[node].G; }
void egso_set_rows(egso *o, int node, const int64_t *core, const int64_t *mem) {
  node_t *nd = &o->nodes[node];
  for (int i = 0; i < nd->G; i++) { nd->g[i].ca = core[i]; nd->g[i].ma = mem[i]; }
}
void egso_get_rows(egso *o, int node, int64_t *core, int64_t *mem) {
  node_t *nd = &o->nodes[node];
  for (int i = 0; i < nd->G; i++) { core[i] = nd->g[i].ca; mem[i] = nd->g[i].ma; }
}
static void opt_export(const opt_t *op, int C, int32_t *off, int32_t *idx) {
  if (!off) return;
  int k = 0;
  for (int i = 0; i < C; i++) {
    off[i] = k;
    for (int j = 0; j < op->n[i]; j++) { if (idx) idx[k] = op->idx[i][j]; k++; }
  }
  off[C] = k;
}
static int opt_import(opt_t *op, int C, const int32_t *off, const int32_t *idx, int G) {
  memset(op, 0, sizeof *op);
  op->C = C;
  for (int i = 0; i < C; i++) {
    int n = off ? off[i + 1] - off[i] : 0;
    if (n < 0 || n > EGSO_MAX_G) return 0;
    op->n[i] = (int8_t)n;
    for (int j = 0; j < n; j++) {
      int v = idx[off[i] + j];
      if (v < 0 || v >= G) return 0; /* the reference would panic (index out of range) */
      op->idx[i][j] = (int8_t)v;
    }
  }
  return 1;
}
int egso_trade(egso *o, int node, int C, const egso_unit *units, int32_t *alloc_off, int32_t *alloc_idx,
               int64_t *score) {
  node_t tmp = o->nodes[node];
  opt_t op;
  if (!trade(o->policy, &tmp, C, units, &op)) return ST_NOFIT;
  opt_export(&op, C, alloc_off, alloc_idx);
  if (score) *score = op.score;
  return ST_OK;
}
int egso_filter(egso *o, int n, const int32_t *node_ids, int C, const egso_unit *units, int threads,
                uint8_t *out_fit) {
  uint32_t shape = intern(o, C, units);
  if (threads <= 1) { filter_range(o, 0, n, node_ids, shape, C, units, out_fit); return ST_OK; }
  pool_t *p = pool_get(o, threads);
  p->n = n; p->ids = node_ids; p->shape = shape; p->C = C; p->u = units; p->fit = out_fit;
  atomic_store(&p->next, 0); atomic_store(&p->done, 0);
  atomic_fetch_add_explicit(&p->gen, 1, memory_order_release);
  pool_work(p);
  while (atomic_load_explicit(&p->done, memory_order_acquire) < threads - 1) { /* wg.Wait(), scheduler.go:156 */ }
  return ST_OK;
}
/* GPUUnitScheduler.Score scheduler.go:170-184 + NodeAllocator.Score node.go:75-85 */
int egso_score(egso *o, int n, const int32_t *node_ids, int C, const egso_unit *units, int64_t *out_score) {
  uint32_t shape = intern(o, C, units);
  int rc = ST_OK;
  for (int i = 0; i < n; i++) {
    int nid = node_ids ? node_ids[i] : i;
    if (nid < 0 || nid >= o->nn || o->nodes[nid].G == 0) { out_score[i] = 0; continue; } /* scheduler.go:176-179 */
    node_t *nd = &o->nodes[nid];
    opt_t *op = cache_find(nd, node_key(o, shape, C, units));
    if (!op) {
      if (node_assume(o, nd, shape, C, units) == NULL) { out_score[i] = 0; continue; } /* node.go:79-82 */
      rc = ST_PANIC; out_score[i] = 0; continue;                                         /* node.go:84 nil deref */
    }
    out_score[i] = op->score;
  }
  return rc;
}
/* NodeAllocator.Add node.go:148-160 */
static int node_add(node_t *nd, int C, const egso_unit *u, const opt_t *op, uint64_t uid) {
  if (pods_has(nd, uid)) return 1;
  pods_add(nd, uid);
  return transact(nd, C, u, op);
}
int egso_bind(egso *o, int node, int C, const egso_unit *units, uint64_t uid, int32_t *alloc_off,
              int32_t *alloc_idx) {
  if (node < 0 || node >= o->nn || o->nodes[node].G == 0) return ST_BAD_ARG;
  uint32_t shape = intern(o, C, units);
  node_t *nd = &o->nodes[node];
  uint32_t key = node_key(o, shape, C, units);
  opt_t *hit = cache_find(nd, key);
  if (!hit) return ST_NO_OPTION;                 /* node.go:93-96 (delete of a missing key is a no-op) */
  opt_t op = *hit;
  cache_del(nd, key);                            /* deferred delete, node.go:90-92 */
  if (!node_add(nd, C, units, &op, uid)) return ST_TRANSACT;
  opt_export(&op, C, alloc_off, alloc_idx);
  set_add(&o->pod_maps, uid);                    /* scheduler.go:224 */
  return ST_OK;
}
int egso_peek(egso *o, int node, int C, const egso_unit *units, int64_t *score, int32_t *alloc_off,
              int32_t *alloc_idx) {
  uint32_t shape = intern(o, C, units);
  opt_t *hit = cache_find(&o->nodes[node], node_key(o, shape, C, units));
  if (!hit) return 0;
  if (score) *score = hit->score;
  opt_export(hit, C, alloc_off, alloc_idx);
  return 1;
}
/* TEST SUPPORT: install cached options of one request shape on nodes [0, n) (node_ids NULL) -- the state of a
 * scheduler that already ran: entry i exists when valid[i] != 0, with option.Score = score[i] and
 * option.Allocated rebuilt from alloc_mask[i][c] (bit g = GPU g of container c; Trade only yields
 * ascending index lists).  Existing entries of that shape on those nodes are replaced. */
int egso_cache_load(egso *o, int C, const egso_unit *units, int n, const int32_t *node_ids,
                    const uint8_t *valid, const int64_t *score, const uint8_t *alloc_mask) {
  if (C < 1 || C > 4) return ST_BAD_ARG;
  uint32_t shape = intern(o, C, units);
  uint32_t key = node_key(o, shape, C, units);
  for (int i = 0; i < n; i++) {
    int node = node_ids ? node_ids[i] : i;
    if (node < 0 || node >= o->nn) return ST_BAD_ARG;
    node_t *nd = &o->nodes[node];
    cache_del(nd, key);
    if (!valid[i]) continue;
    opt_t op; memset(&op, 0, sizeof op);
    op.key = key; op.C = C; op.score = score[i];
    for (int c = 0; c < C; c++) {
      int k = 0;
      for (int g = 0; g < 8; g++) if ((alloc_mask[(size_t)i * 4 + c] >> g) & 1) op.idx[c][k++] = (int8_t)g;
      op.n[c] = (int8_t)k;
    }
    cache_put(nd, &op);
  }
  return ST_OK;
}
/* TEST SUPPORT: the inverse of egso_cache_load, egso_peek over nodes [0, n) in one call: valid[i] = 1 when node i
 * holds an entry of the shape, then score[i] and alloc_mask[i][c] as egso_cache_load takes them (0 otherwise). */
int egso_cache_dump(egso *o, int C, const egso_unit *units, int n, uint8_t *valid, int64_t *score, uint8_t *alloc_mask) {
  if (C < 1 || C > 4 || n < 0 || n > o->nn) return ST_BAD_ARG;
  uint32_t shape = intern(o, C, units);
  uint32_t key = node_key(o, shape, C, units);
  for (int i = 0; i < n; i++) {
    opt_t *hit = cache_find(&o->nodes[i], key);
    valid[i] = hit != NULL;
    score[i] = hit ? hit->score : 0;
    for (int c = 0; c < 4; c++) {
      uint8_t m = 0;
      if (hit && c < C)
        for (int k = 0; k < hit->n[c]; k++) m |= (uint8_t)(1u << hit->idx[c][k]);
      alloc_mask[(size_t)i * 4 + c] = m;
    }
  }
  return ST_OK;
}
/* AddPod scheduler.go:229-245 */
int egso_add_pod(egso *o, int node, int C, const egso_unit *units, const int32_t *alloc_off,
                 const int32_t *alloc_idx, uint64_t uid) {
  if (node < 0 || node >= o->nn || o->nodes[node].G == 0) return ST_BAD_ARG;
  if (set_has(&o->pod_maps, uid)) return ST_OK;
  opt_t op;
  if (!opt_import(&op, C, alloc_off, alloc_idx, o->nodes[node].G)) return ST_BAD_ARG;
  node_add(&o->nodes[node], C, units, &op, uid); /* error discarded, scheduler.go:242 */
  set_add(&o->pod_maps, uid);
  return ST_OK;
}
/* ForgetPod scheduler.go:247-267 + NodeAllocator.Forget node.go:129-140 */
int egso_forget_pod(egso *o, int node, int C, const egso_unit *units, const int32_t *alloc_off,
                    const int32_t *alloc_idx, uint64_t uid) {
  if (node >= 0) {
    if (node >= o->nn || o->nodes[node].G == 0) return ST_BAD_ARG;
    node_t *nd = &o->nodes[node];
    if (pods_has(nd, uid)) {
      opt_t op;
      if (!opt_import(&op, C, alloc_off, alloc_idx, nd->G)) return ST_BAD_ARG;
      cancel(nd, C, units, &op);
      pods_del(nd, uid);
    }
  }
  if (set_has(&o->pod_maps, uid)) { set_del(&o->pod_maps, uid); set_add(&o->released, uid); }
  return ST_OK;
}
int egso_known_pod(egso *o, uint64_t uid) { return set_has(&o->pod_maps, uid); }
int egso_released_pod(egso *o, uint64_t uid) { return set_has(&o->released, uid); }

int egso_schedule_batch(egso *o, int P, const int32_t *c_off, const egso_unit *units, const uint64_t *uids,
                        int threads, int32_t *out_node, int32_t *out_status, uint8_t *out_alloc_mask,
                        int32_t *out_fit_count, uint64_t *out_fit_digest, uint64_t *out_score_digest,
                        int vec_pods, uint8_t *vec_fit, int32_t *vec_score) {
  int N = o->nn;
  uint8_t *fit = malloc((size_t)N > 0 ? (size_t)N : 1);
  int32_t *ids = malloc(sizeof(int32_t) * (size_t)(N > 0 ? N : 1));
  int64_t *sc = malloc(sizeof(int64_t) * (size_t)(N > 0 ? N : 1));
  for (int p = 0; p < P; p++) {
    int C = c_off[p + 1] - c_off[p];
    const egso_unit *u = units + c_off[p];
    egso_filter(o, N, NULL, C, u, threads, fit);                 /* /scheduler/filter  */
    int nf = 0;
    for (int i = 0; i < N; i++) if (fit[i]) ids[nf++] = i;       /* filteredNodes, input order (scheduler.go:158-167) */
    egso_score(o, nf, ids, C, u, sc);                            /* /scheduler/priorities */
    uint64_t fd = 0, sd = 0;
    int w = -1; int64_t best = 0;
    for (int j = 0; j < nf; j++) {
      fd += egso_mix64(2ull * (uint64_t)ids[j] + 1);
      sd += egso_mix64(2ull * (uint64_t)ids[j] + 2) * (2ull * (uint64_t)(uint32_t)(int32_t)sc[j] + 1);
      if (w < 0 || sc[j] > best) { w = ids[j]; best = sc[j]; }   /* first max */
    }
    if (p < vec_pods) {
      if (vec_fit) memcpy(vec_fit + (size_t)p * N, fit, (size_t)N);
      if (vec_score) {
        int32_t *row = vec_score + (size_t)p * N;
        memset(row, 0, sizeof(int32_t) * (size_t)N);
        for (int j = 0; j < nf; j++) row[ids[j]] = (int32_t)sc[j];
      }
    }
    int st = ST_NOFIT;
    uint8_t mask[4] = {0, 0, 0, 0};
    if (w >= 0) {
      int32_t off[EGSO_MAX_C + 1], idx[EGSO_MAX_C * EGSO_MAX_G];
      st = egso_bind(o, w, C, u, uids ? uids[p] : (uint64_t)p, off, idx); /* /scheduler/bind */
      if (st == ST_OK)
        for (int c = 0; c < C && c < 4; c++)
          for (int k = off[c]; k < off[c + 1]; k++) if (idx[k] < 8) mask[c] |= (uint8_t)(1u << idx[k]);
    }
    if (out_node) out_node[p] = w;
    if (out_status) out_status[p] = st;
    if (out_alloc_mask) memcpy(out_alloc_mask + 4 * (size_t)p, mask, 4);
    if (out_fit_count) out_fit_count[p] = nf;
    if (out_fit_digest) out_fit_digest[p] = fd;
    if (out_score_digest) out_score_digest[p] = sd;
  }
  free(fit); free(ids); free(sc);
  return P;
}
