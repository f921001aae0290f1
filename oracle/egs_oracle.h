/*
 * egs_oracle.h -- CPU ORACLE: TEST INFRASTRUCTURE ONLY.
 *
 * A plain-C restatement of the reference's Filter/Score/Allocate path
 * (pkg/scheduler/{gpu,rater,allocate,node,scheduler}.go).  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may link or call it; libegs never does.
 *
 * PARITY STATUS: "parity unpinned" -- the reference's own test has no assertions
 * (pkg/scheduler/scheduler_test.go:11-24) and no Go toolchain exists here; the
 * pins are SURVEY.md 8c's hand-traced vectors (tests/test_oracle_ka.py) and the
 * sha256 KATs of R8.
 */
#ifndef EGS_ORACLE_H_
#define EGS_ORACLE_H_
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define EGSO_MAX_G 16
#define EGSO_MAX_C 8

typedef struct egso egso;
typedef struct { int64_t core, mem, count; } egso_unit;   /* GPUUnit, gpu.go:9-13 (Go int = 64 bit) */

/* policy 0 = binpack, 1 = spread; faithful != 0 re-formats + sha256-hashes the request
 * per node per verb like node.go:62-63,76-77,88-89 (cache keyed by the 8-hex prefix). */
egso *egso_create(int policy, int faithful);
void egso_destroy(egso *o);
/* NewNodeAllocator (node.go:23-59); returns the dense node id, or -1 ("no gpu available"). */
int egso_add_node(egso *o, int64_t core_allocatable, int64_t mem_allocatable);
int egso_num_nodes(egso *o);
int egso_gpu_count(egso *o, int node);
void egso_set_rows(egso *o, int node, const int64_t *core, const int64_t *mem);
void egso_get_rows(egso *o, int node, int64_t *core, int64_t *mem);

/* GPURequest.Hash (allocate.go:30-33) -> 8 hex chars + NUL */
void egso_request_hash(int C, const egso_unit *units, char out[9]);
/* NewGPURequest for one container (allocate.go:38-53) */
void egso_unit_from_requests(int64_t core, int64_t mem, egso_unit *out);

/* GPUs.Trade on a scratch copy of the node's rows (gpu.go:65-129): no cache effects.
 * alloc_off[C+1]/alloc_idx give Allocated; returns 0 ok / 1 nofit. */
int egso_trade(egso *o, int node, int C, const egso_unit *units,
               int32_t *alloc_off, int32_t *alloc_idx, int64_t *score);

/* Assume (scheduler.go:112-168): threads<=1 serial; otherwise that many workers drain
 * the node indices (4 in the reference, scheduler.go:135). */
int egso_filter(egso *o, int n, const int32_t *node_ids, int C, const egso_unit *units,
                int threads, uint8_t *out_fit);
/* Score (scheduler.go:170-184): serial.  Returns 9 if the reference would panic. */
int egso_score(egso *o, int n, const int32_t *node_ids, int C, const egso_unit *units,
               int64_t *out_score);
/* Bind -> Allocate (scheduler.go:186-199, node.go:87-104). */
int egso_bind(egso *o, int node, int C, const egso_unit *units, uint64_t uid,
              int32_t *alloc_off, int32_t *alloc_idx);
int egso_peek(egso *o, int node, int C, const egso_unit *units, int64_t *score,
              int32_t *alloc_off, int32_t *alloc_idx);   /* 1 = cached */
int egso_add_pod(egso *o, int node, int C, const egso_unit *units,
                 const int32_t *alloc_off, const int32_t *alloc_idx, uint64_t uid);
int egso_forget_pod(egso *o, int node, int C, const egso_unit *units,
                    const int32_t *alloc_off, const int32_t *alloc_idx, uint64_t uid);
/* TEST SUPPORT: load cached options of one shape (a scheduler that already ran); see egs_oracle.c */
int egso_cache_load(egso *o, int C, const egso_unit *units, int n, const int32_t *node_ids,
                    const uint8_t *valid, const int64_t *score, const uint8_t *alloc_mask);
int egso_cache_dump(egso *o, int C, const egso_unit *units, int n, uint8_t *valid, int64_t *score, uint8_t *alloc_mask);
int egso_known_pod(egso *o, uint64_t uid);
int egso_released_pod(egso *o, uint64_t uid);

/* Driver rule over ALL nodes in index order (SURVEY.md 8d).  Pod p = units[c_off[p]..c_off[p+1]).
 * out_alloc_mask is [P][4] (containers beyond 4 and GPUs beyond 8 are not representable: 0).
 * vec_fit / vec_score, when non-NULL, receive the full per-pod vectors ([P][N], score of unfit = 0)
 * for pods [0, vec_pods).  Returns the number of pods processed. */
int egso_schedule_batch(egso *o, int P, const int32_t *c_off, const egso_unit *units,
                        const uint64_t *uids, int threads,
                        int32_t *out_node, int32_t *out_status, uint8_t *out_alloc_mask,
                        int32_t *out_fit_count, uint64_t *out_fit_digest, uint64_t *out_score_digest,
                        int vec_pods, uint8_t *vec_fit, int32_t *vec_score);

uint64_t egso_mix64(uint64_t x);
void egso_sha256(const uint8_t *msg, uint64_t len, uint8_t out[32]);

#ifdef __cplusplus
}
#endif
#endif
