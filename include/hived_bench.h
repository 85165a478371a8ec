/* hived_bench.h — measurement hooks exported by libhived_cuda.so next to the ABI of hived.h.
 * They exist so that bench.py can (a) time the kernel with the batch already resident in HBM and
 * (b) rewind the scheduler state between timed steps.  Not part of the reference-facing surface. */
#ifndef HIVED_BENCH_H_
#define HIVED_BENCH_H_
#include "hived.h"
#ifdef __cplusplus
extern "C" {
#endif
int hived_bench_save_state(hived_ctx*);     /* device-to-device copy of every mutable array */
int hived_bench_restore_state(hived_ctx*);
int hived_bench_stage_events(hived_ctx*, const hived_event_t* events, int32_t n, int64_t pool_cap); /* H2D once */
int hived_bench_run_staged(hived_ctx*);     /* one kernel launch over the staged batch; nothing crosses PCIe */
int hived_bench_fetch_results(hived_ctx*, hived_result_t* res, int32_t* pool, int64_t pool_cap, int64_t* pool_used);
int hived_bench_flush_l2(hived_ctx*);       /* overwrite a buffer larger than L2 */
/* out[0..15): SM cycles of the leader warps in {view pass, leaf search, v->p mapping, result emission, commit, delete,
 * all events, waiting at shared sections}, the number of shared sections entered, then cycles / events of
 * {Schedule of a pod of an existing gang, delete of a pod that is not the gang's last, commit of such a pod} */
int hived_bench_phase_cycles(hived_ctx*, int64_t* out);
int hived_bench_debug_cycles(hived_ctx*, int64_t* out); /* out[0..16): scratch cycle counters used in profiling sessions */
/* out[0..12): events by path — [0] scheduling passes answered by the bucketed cluster view, [1] full view passes,
   [2] bucket rebuilds, [3] nodes moved between buckets, [4]/[5] gang commits fast/general, [6]/[7] gang releases
   fast/general, [8]/[9] virtual->physical mappings fast/general; returns the number of counters */
int hived_bench_path_counters(hived_ctx*, int64_t* out);
double hived_bench_last_kernel_ms(hived_ctx*);   /* CUDA-event time of the last launch, on its stream */
double hived_bench_total_kernel_ms(hived_ctx*);
int64_t hived_bench_kernel_launches(hived_ctx*);
int hived_bench_num_ctas(hived_ctx*);            /* CTAs the last batch ran on (VC-parallel execution) */
int hived_bench_set_result_hash(hived_ctx*, int on); /* toggle the running parity hash (HIVED_OPT_NO_RESULT_HASH) */

/* Test hooks: scheduler state that no result or cell snapshot shows but that decides later calls, for comparing two
 * implementations of hived.h call by call.  Both are host-side reads of the state; neither changes it. */
uint64_t hived_debug_view_hash(hived_ctx*); /* hash of every cluster view's persisted order */
/* Fills out[0..min(cap, n)) and returns n, the number of int32 words of the canonical encoding: a sequence of
 * sections, each starting with its tag, in this order (cells / nodes / VCs / chains are ABI ids, levels 1-based;
 * empty lists, zero counters and missing map entries are omitted):
 *   FREE        chain level n cell*n          free cell list, in slice order, duplicates included
 *   BAD_FREE    chain level n cell*n          bad free cells
 *   DOOMED_BAD  vc chain level n cell*n       a VC's doomed bad cells
 *   VC_FREE     vc chain level count          only (vc, chain) pairs the VC has a counter for
 *   ALL_VC_FREE / TOTAL_LEFT / ALL_VC_DOOMED  chain level count
 *   USED_PHYSICAL / USED_VIRTUAL  cell n (priority count)*n   used leaf cells per priority, ascending priority
 *   USING_GROUP / RESERVING_GROUP cell group live  a physical cell's group; live = 0: not the object its name maps to
 *   BAD_NODE    node */
enum {
  HIVED_DS_FREE = 1, HIVED_DS_BAD_FREE = 2, HIVED_DS_DOOMED_BAD = 3, HIVED_DS_VC_FREE = 4, HIVED_DS_ALL_VC_FREE = 5,
  HIVED_DS_TOTAL_LEFT = 6, HIVED_DS_ALL_VC_DOOMED = 7, HIVED_DS_USED_PHYSICAL = 8, HIVED_DS_USED_VIRTUAL = 9,
  HIVED_DS_USING_GROUP = 10, HIVED_DS_RESERVING_GROUP = 11, HIVED_DS_BAD_NODE = 12
};
int64_t hived_debug_state(hived_ctx*, int32_t* out, int64_t cap);
#ifdef __cplusplus
}
#endif
#endif
