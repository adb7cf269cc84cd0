/*
 * pinot_b200.h — C ABI of libpinot_b200.so, the B200-native executor for Apache Pinot's per-segment
 * scan -> filter -> project -> group-by/aggregate path.
 *
 * This is the boundary a JNI shim binds (jni/pinot_b200_jni.c, INTEGRATION.md).  Plain pointers and
 * sizes only.  Every entry point names the reference interface it stands in for
 * (CTR  = pinot-core/src/main/java/org/apache/pinot/core,
 *  SEGL = pinot-segment-local/src/main/java/org/apache/pinot/segment/local,
 *  SPI  = pinot-segment-spi/src/main/java/org/apache/pinot/segment/spi).
 *
 * Division of labour (SURVEY.md §8b): the host side (Java in a Pinot server; pinot_b200/csrc/host in
 * this repo) runs the reference's own PredicateEvaluator lowering and FilterOperatorUtils index
 * selection, and hands over (a) the segment's index buffers exactly as mmap'd and (b) a filter tree
 * whose leaves are already in dictId / docId-range / bitmap form.  Everything per-row happens on the GPU.
 *
 * Threading: all functions are thread-safe; one call = one CUDA stream.  Errors: 0 = PB_OK, negative
 * code otherwise with a thread-local message in pb_last_error().  The library never aborts and never
 * falls back to a CPU implementation.
 */
#ifndef PINOT_B200_H
#define PINOT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_OK 0
#define PB_ERR_INVALID (-1)       /* malformed descriptor */
#define PB_ERR_UNSUPPORTED (-2)   /* outside the eligible set: the plan maker must decline to the CPU plan */
#define PB_ERR_CUDA (-3)
#define PB_ERR_OOM (-4)
#define PB_ERR_STATE (-5)

/* FieldSpec.DataType stored types (pinot-spi/.../data/FieldSpec.java) on this path */
enum { PB_INT = 0, PB_LONG = 1, PB_FLOAT = 2, PB_DOUBLE = 3, PB_STRING = 4 };

/* AggregationFunctionType subset (CTR/query/aggregation/function) */
enum { PB_AGG_COUNT = 0, PB_AGG_SUM = 1, PB_AGG_MIN = 2, PB_AGG_MAX = 3, PB_AGG_AVG = 4, PB_AGG_DISTINCTCOUNT = 5 };

/* Filter tree node kinds.  Leaves are the OUTPUT of PredicateEvaluator + FilterOperatorUtils:
 *   SCAN_*      ScanBasedFilterOperator  (CTR/operator/filter/ScanBasedFilterOperator.java:59-66)
 *   INVERTED    InvertedIndexFilterOperator (…/InvertedIndexFilterOperator.java:60-96)
 *   SORTED      SortedIndexBasedFilterOperator (…/SortedIndexBasedFilterOperator.java:53-131)
 *   BITMAP      BitmapBasedFilterOperator (…/BitmapBasedFilterOperator.java:42-60), e.g. upsert validDocIds
 *   AND/OR/NOT  And/Or/NotFilterOperator */
enum {
  PB_F_AND = 0, PB_F_OR = 1, PB_F_NOT = 2, PB_F_MATCH_ALL = 3, PB_F_EMPTY = 4,
  PB_F_SCAN_DICT_RANGE = 5,   /* dictionary column, lo <= dictId < hi                                   */
  PB_F_SCAN_DICT_SET = 6,     /* dictionary column, dictId in ids[] (exclusive: NOT in)                 */
  PB_F_SCAN_RAW_RANGE = 7,    /* raw column: INT/LONG lo..hi inclusive; FLOAT/DOUBLE dlo..dhi + flags   */
  PB_F_SCAN_RAW_SET = 8,      /* raw column: value in raw_values[] (exclusive: NOT in); doubles as bits */
  PB_F_INVERTED = 9,          /* bitmap inverted index: OR of the bitmaps of ids[] (exclusive: flipped) */
  PB_F_SORTED = 10,           /* sorted index: ids[] holds num_ids inclusive (start,end) docId pairs    */
  PB_F_BITMAP = 11            /* RoaringBitmap portable blob (exclusive: flipped); blob NULL = `column`'s null_value_vector (IS [NOT] NULL) */
};

typedef struct pb_segment_s* pb_segment_handle;
typedef struct pb_group_s* pb_segment_group_handle;
typedef struct pb_result_s* pb_result_handle;

/* One column's index buffers, exactly as sliced out of columns.psf
 * (SPI/store/SegmentDirectory.java:179 getIndexFor; big-endian Pinot layouts, SURVEY.md Appendix A). */
typedef struct pb_column_desc {
  const char* name;
  int32_t stored_type;         /* PB_INT .. PB_STRING */
  int32_t has_dictionary;
  int32_t is_sorted;
  int32_t cardinality;         /* column.<name>.cardinality (dictionary columns) */
  int32_t bits_per_element;    /* column.<name>.bitsPerElement */
  int32_t dict_entry_bytes;    /* 4/8 for numerics, lengthOfEachEntry for STRING */
  const void* forward_index;   /* .sv.unsorted.fwd | .sv.sorted.fwd | .sv.raw.fwd (fixed-width values; chunks PASS_THROUGH, or SNAPPY /
                                * LZ4 / LZ4_LENGTH_PREFIXED compressed: those are decoded on the device when the column is staged) */
  uint64_t forward_index_len;
  const void* dictionary;      /* .dict, NULL for raw columns */
  uint64_t dictionary_len;
  const void* inverted_index;  /* .bitmap.inv, NULL when absent */
  uint64_t inverted_index_len;
  const void* null_value_vector;   /* .bitmap.nullvalue (DataSource.getNullValueVector(): one RoaringBitmap of the null docIds), NULL when
                                    * absent.  Only IS NULL / IS NOT NULL read it (FilterPlanNode.java:294-307); queries with
                                    * enableNullHandling keep the CPU plan */
  uint64_t null_value_vector_len;
} pb_column_desc;

typedef struct pb_segment_desc {
  const char* segment_name;
  int32_t num_docs;            /* segment.total.docs */
  int32_t num_columns;
  const pb_column_desc* columns;
} pb_segment_desc;

typedef struct pb_filter_node {
  int32_t kind;                /* PB_F_* */
  int32_t column;              /* index into pb_segment_desc.columns (leaves on a column) */
  int32_t num_children;        /* AND / OR: operand count (postfix); NOT: 1 */
  int32_t exclusive;           /* NEQ / NOT_IN semantics for *_SET, INVERTED, BITMAP */
  int64_t lo, hi;              /* SCAN_DICT_RANGE: [lo,hi) dictIds; SCAN_RAW_RANGE (INT/LONG): [lo,hi] */
  double dlo, dhi;             /* SCAN_RAW_RANGE (FLOAT/DOUBLE) */
  int32_t dlo_inclusive, dhi_inclusive;
  const int32_t* ids;          /* dictIds (sorted ascending) or docId pairs */
  int32_t num_ids;
  int32_t num_raw_values;
  const int64_t* raw_values;   /* SCAN_RAW_SET: INT/LONG values; FLOAT/DOUBLE as IEEE-754 double bits */
  const void* blob;            /* PB_F_BITMAP */
  uint64_t blob_len;
} pb_filter_node;

/* Per-segment part of a query: the filter in postfix order (empty = match all).  It is per segment
 * because dictIds are segment-local (FilterPlanNode.run is per segment: CTR/plan/FilterPlanNode.java:88-106). */
typedef struct pb_segment_query {
  const pb_filter_node* filter;
  int32_t num_filter_nodes;
  /* Filtered aggregations (FilteredGroupByOperator / FilteredAggregationOperator, CTR/operator/query/
   * FilteredGroupByOperator.java:108-159): the FILTER(WHERE ...) clause f of the query, lowered for this segment,
   * is agg_filters[f] with agg_filter_nodes[f] postfix nodes (0 nodes = matches all).  pb_query_desc.num_agg_filters
   * entries; both pointers may be NULL when that is 0. */
  const pb_filter_node* const* agg_filters;
  const int32_t* agg_filter_nodes;
} pb_segment_query;

typedef struct pb_aggregation_desc {
  int32_t op;                  /* PB_AGG_* */
  const char* column;          /* NULL for COUNT(*) */
} pb_aggregation_desc;

typedef struct pb_order_by {
  int32_t kind;                /* 0 = the index-th group-by column, 1 = the index-th aggregation (COUNT / SUM / MIN / MAX / AVG) */
  int32_t index;
  int32_t descending;
} pb_order_by;

#define PB_Q_COMBINE 1u            /* one merged table over all segments (GroupByCombineOperator semantics, on device) */
#define PB_Q_DEFER_FINALIZE 2u     /* leave tables on the device for a cross-GPU reduce; call pb_result_finalize */
#define PB_Q_GENERIC_KERNEL 4u     /* force the width-generic predicate path (testing / A-B measurement) */
#define PB_Q_GATHER_IN_PLACE 16u   /* cold segments: columns that are only gathered (group-by keys, aggregation inputs) and are not
                                    * resident in HBM yet are read in place from the caller's pb_host_register'd buffers (a few
                                    * PCIe sectors per matching row) instead of being copied whole; predicate columns are staged.
                                    * Buffers that are not page-locked/mapped or not 4-byte aligned are staged as usual. */
#define PB_Q_NO_TMA 8u             /* stage tiles with ld.global/st.shared instead of cp.async.bulk (testing) */
#define PB_Q_ALL_RANKS 32u         /* collective call (needs PB_Q_COMBINE and pb_comm_init): every rank runs the same query over its own
                                    * segments, the per-rank tables are merged over NCCL on the call's stream inside the library
                                    * (all-gather of the table block + one merge kernel; hash tables: hash-partitioned all-to-all),
                                    * and every rank gets the merged result.  The ranks must agree on the global dictionaries of the
                                    * group-by / DISTINCTCOUNT columns first (pb_segment_group_export_dictionary /
                                    * _set_global_dictionary) and must issue their PB_Q_ALL_RANKS calls in the same order. */
#define PB_Q_NULL_HANDLING 64u     /* the query runs with enableNullHandling (QueryContext.isNullHandlingEnabled): the caller has folded the
                                    * three-valued filter into its "trues" program (BaseFilterOperator.getTrues / getFalses) and given
                                    * every aggregation over a nullable column the implicit clause "<column> IS NOT NULL" as its FILTER
                                    * clause (NullableSingleInputAggregationFunction.java:72-134 skips null docs) -- pbh_execute does both.
                                    * The device then keeps the row count of EVERY aggregation (pb_result_long: COUNT value, AVG
                                    * denominator, and for SUM / MIN / MAX the number of non-null inputs): 0 means the function's result
                                    * is SQL NULL for that group */

typedef struct pb_query_desc {
  int32_t num_group_by;
  const char* const* group_by_columns;
  int32_t num_aggregations;
  const pb_aggregation_desc* aggregations;
  int32_t num_groups_limit;                     /* InstancePlanMakerImplV2.java:79 (default 100000) */
  int32_t max_initial_result_holder_capacity;   /* InstancePlanMakerImplV2.java:70 (default 10000) */
  uint32_t flags;                               /* PB_Q_* */
  /* filtered aggregations: number of distinct FILTER(WHERE ...) clauses (<= 8) and, per aggregation, the index of its
   * clause (-1 = none; NULL when num_agg_filters = 0).  QueryContext.getFilteredAggregationFunctions(). */
  int32_t num_agg_filters;
  const int32_t* agg_filter_of;
  /* ORDER BY ... LIMIT trim of a group-by result, on the device (the combine layer's server-side trim: IndexedTable +
   * TableResizer keep trim_size = max(5 x LIMIT, minServerGroupTrimSize) groups once a table holds more than
   * trim_threshold = groupTrimThreshold groups; CTR/util/GroupByUtils.java:44-70, CTR/data/table/TableResizer.java).
   * order_by[0] selects: the trim_size best groups by it survive, plus every group that ties with the last of them; further
   * ORDER BY expressions are left to the broker's final sort.  num_order_by = 0 or trim_size <= 0: no trim. */
  int32_t num_order_by;
  const struct pb_order_by* order_by;
  int32_t trim_size;
  int32_t trim_threshold;
} pb_query_desc;

/* ExecutionStatistics (CTR/operator/ExecutionStatistics.java:28-65) */
typedef struct pb_exec_stats {
  int64_t num_docs_scanned;
  int64_t num_entries_scanned_in_filter;
  int64_t num_entries_scanned_post_filter;
  int64_t num_total_docs;
  int32_t num_groups_limit_reached;
  int32_t num_segments;
} pb_exec_stats;

/* -------- lifecycle -------- */
/* device_ids: the CUDA devices this process drives (NULL / 0 = the calling thread's current device).  Every later entry
 * point selects the device of the handle it works on, so calls may come from any thread (SURVEY.md §8b: nextBlock() runs on
 * the query executor's worker threads, BaseCombineOperator.java:100-141).  hbm_cache_bytes bounds the staged segment data
 * per device (0 = unlimited): least-recently-used segments that no query is using are dropped from HBM and re-staged from
 * the caller's buffers on their next use. */
int pb_init(const int* device_ids, int n_devices, size_t hbm_cache_bytes);
int pb_shutdown(void);
const char* pb_last_error(void);
int pb_device_count(void);

/* -------- multi-GPU.  Two deployments:
 *   (a) one process driving several GPUs (one JVM, pb_init with n_devices > 1): stage each segment on a device_index of
 *       your choice; a query over a group whose segments span devices runs every device's part concurrently and merges the
 *       tables on the first device over NVLink -- nothing else to call.  This is BaseCombineOperator's segment parallelism
 *       (CTR/operator/combine/BaseCombineOperator.java:97-142) across GPUs instead of threads.
 *   (b) one process per GPU (torchrun, or several server JVMs on one box): every process calls pb_comm_init with the same
 *       128-byte id (made by pb_comm_unique_id on one rank and distributed by the caller: a file, a socket, torch.distributed)
 *       and then passes PB_Q_ALL_RANKS to pb_query_execute.  NCCL is loaded at run time (PB_NCCL_LIB overrides the search);
 *       single-GPU servers never need it. -------- */
#define PB_COMM_ID_BYTES 128
int pb_comm_unique_id(void* out, size_t cap);                                     /* ncclGetUniqueId */
int pb_comm_init(int n_ranks, int rank, const void* unique_id, size_t id_bytes);  /* ncclCommInitRank on this process's device */
int pb_comm_info(int* n_ranks, int* rank);                                        /* returns 1 when a communicator exists */
int pb_comm_destroy(void);

/* -------- segment staging: replaces the DataSource / ForwardIndexReader / Dictionary / InvertedIndexReader
 * objects the operators pull from IndexSegment.getDataSource (SPI/datasource/DataSource.java:38-60).
 * Copies the buffers to HBM once; the handle is valid until pb_segment_release. -------- */
int pb_segment_stage(const pb_segment_desc* desc, int device_index, pb_segment_handle* out);
int pb_segment_release(pb_segment_handle seg);
int64_t pb_segment_device_bytes(pb_segment_handle seg);
/* segment cache of one device: bytes staged right now and segments evicted so far (hbm_cache_bytes of pb_init) */
int pb_cache_stats(int device_index, int64_t* staged_bytes, int64_t* evictions);

/* A set of segments queried together.  Holds the per-column global dictionaries (sorted union of the
 * segment dictionaries) and local->global dictId remaps that make a device-side cross-segment merge
 * possible (the reference merges by decoded value: CTR/operator/combine/GroupByCombineOperator.java:132-147). */
int pb_segment_group_create(const pb_segment_handle* segs, int n_segs, pb_segment_group_handle* out);
int pb_segment_group_release(pb_segment_group_handle g);
/* Cross-process agreement on a column's global dictionary (multi-GPU): export this group's union, and
 * install the union over all ranks.  values are native-endian stored-type values (STRING: fixed-width
 * padded entries of entry_bytes each). */
int pb_segment_group_export_dictionary(pb_segment_group_handle g, const char* column, const void** values,
                                       int64_t* num_values, int32_t* entry_bytes);
int pb_segment_group_set_global_dictionary(pb_segment_group_handle g, const char* column, const void* values,
                                           int64_t num_values, int32_t entry_bytes);

/* host view of segment `segment_index`'s local -> global dictId remap for `column` (length = local cardinality) */
int pb_segment_group_remap(pb_segment_group_handle g, const char* column, int32_t segment_index, const int32_t** remap, int32_t* n);

/* -------- execution: replaces GroupByOperator.getNextBlock / AggregationOperator.getNextBlock
 * (CTR/operator/query/GroupByOperator.java:101-140, AggregationOperator.java:64-80) for every segment of
 * the group in one call.  seg_queries[i] belongs to the i-th segment of the group. -------- */
int pb_query_execute(pb_segment_group_handle g, const pb_segment_query* seg_queries, const pb_query_desc* q,
                     pb_result_handle* out);

/* -------- results: the contents of GroupByResultsBlock / AggregationResultsBlock
 * (CTR/operator/blocks/results/GroupByResultsBlock.java:68-139, AggregationGroupByResult.java:31-57).
 * Without PB_Q_COMBINE there is one table per segment (table index = segment index); with it, one.
 * All returned pointers are pinned host memory owned by the result handle. -------- */
int32_t pb_result_num_tables(pb_result_handle r);
int64_t pb_result_num_groups(pb_result_handle r, int32_t table);          /* 1 for keyless aggregation */
/* group key of column gb: dictIds (segment-local without COMBINE, global with it); NULL for raw key columns */
const int32_t* pb_result_group_dict_ids(pb_result_handle r, int32_t table, int32_t gb);
/* decoded key values (GroupKeyGenerator.GroupKey._keys): native-endian stored-type values; STRING keys are
 * fixed-width padded entries.  *stored_type / *entry_bytes describe the array. */
const void* pb_result_group_key_values(pb_result_handle r, int32_t table, int32_t gb, int32_t* stored_type,
                                       int32_t* entry_bytes);
/* per aggregation arrays [num_groups]: SUM/MIN/MAX value, AVG sum -> double; COUNT, AVG count,
 * DISTINCTCOUNT size -> long */
const double* pb_result_double(pb_result_handle r, int32_t table, int32_t agg);
const int64_t* pb_result_long(pb_result_handle r, int32_t table, int32_t agg);
/* DISTINCTCOUNT intermediate value sets (BaseDistinctAggregateAggregationFunction.java:760-806):
 * offsets[num_groups+1] into dictIds (ascending per group; local without COMBINE, global with it) */
const int64_t* pb_result_distinct_offsets(pb_result_handle r, int32_t table, int32_t agg);
const int32_t* pb_result_distinct_dict_ids(pb_result_handle r, int32_t table, int32_t agg);
/* DISTINCTCOUNT on a raw (no-dictionary) column: the value sets as bits, ascending per group (INT / LONG: the value;
 * FLOAT / DOUBLE: IEEE-754 bits of the value widened to double); same offsets.  NULL for dictionary columns. */
const int64_t* pb_result_distinct_values(pb_result_handle r, int32_t table, int32_t agg);
const pb_exec_stats* pb_result_stats(pb_result_handle r, int32_t table);
/* device time (CUDA events on the call's stream): the whole call (table init .. result read-back), the two hot
 * kernels together (pb_filter_kernel + pb_agg_kernel), and each of them */
double pb_result_device_ms(pb_result_handle r);
double pb_result_scan_kernel_ms(pb_result_handle r);
int pb_result_phase_ms(pb_result_handle r, double* filter_kernel_ms, double* agg_kernel_ms);
int32_t pb_result_kernel_launches(pb_result_handle r);
double pb_result_comm_ms(pb_result_handle r);           /* device time of the cross-rank merge (collective + merge kernel) */
int32_t pb_result_in_place_columns(pb_result_handle r);   /* (segment, column) pairs this query gathered in place from host memory */
int32_t pb_result_residual_leaves(pb_result_handle r);    /* (segment, filter leaf) pairs the aggregation kernel tested on its rows */
/* host-side microseconds spent in this call, by phase: [0] resolve + stage, [1] table allocation + init,
 * [2] descriptor build + upload, [3] kernel launches, [4] wait for the scan + group count, [5] compaction,
 * gathers and read-back, [6] host key decode / stats; [7] reserved */
int pb_result_host_timing(pb_result_handle r, double* out8);
void pb_result_free(pb_result_handle r);

/* -------- multi-GPU (PB_Q_COMBINE | PB_Q_DEFER_FINALIZE): device-resident table arrays for an
 * NCCL all-reduce issued by the caller (torch.distributed), then finalize on the root.
 * which: 0 = row counts (int64, SUM); 1 = per-aggregation double sums (float64, SUM);
 *        2 = per-aggregation min/max in order-preserving int64 encoding (int64; reduce with MIN for both:
 *            MAX tables hold the bit-complement);
 *        5 / 6 / 7 = the same data as three contiguous spans, one collective each: 5 = counters + row counts
 *            (int64, SUM), 6 = all sums (float64, SUM; may be empty), 7 = all min/max tables (int64, MIN; may be empty);
 *        3 = per-aggregation distinct bitset words (int32; OR == MAX over 0/1 is NOT valid — all-gather + pb_or) -------- */
int pb_result_device_buffer(pb_result_handle r, int32_t which, int32_t agg, void** device_ptr, int64_t* num_elements);
/* which = 8: the whole reducible state of the table as one byte block (num_elements = bytes).  all-gather it across
 * ranks (one collective) and hand the rank-major copies to pb_result_merge_gathered, which reduces them into this result on
 * the result's stream with the right operator per region (u64 SUM | f64 SUM | bitset OR | i64 MIN) — this also merges
 * DISTINCTCOUNT bitsets, which no NCCL reduction operator can. */
int pb_result_merge_gathered(pb_result_handle r, const void* gathered_device_ptr, int32_t n_ranks);
int pb_result_finalize(pb_result_handle r);
/* the CUDA stream (cudaStream_t) this result's work was issued on, and a host-side wait for it */
void* pb_result_stream(pb_result_handle r);
int pb_result_wait(pb_result_handle r);

/* Page-lock a caller-owned buffer (e.g. the mmap'd columns.psf of a segment) so staging runs at full PCIe
 * rate; optional.  Wraps cudaHostRegister / cudaHostUnregister. */
int pb_host_register(const void* ptr, size_t bytes);   /* cudaHostRegisterPortable | cudaHostRegisterMapped */
int pb_host_unregister(const void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* PINOT_B200_H */
