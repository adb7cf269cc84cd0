// pb_device.cuh — device-side data model and kernels of the B200 segment executor (sm_100a).
//
// Two kernels run the per-segment operator chain for every segment of a query in one launch each
// (reference: CTR/operator/query/GroupByOperator.java:101-140 and the call stack in SURVEY.md §3.1):
//
//   pb_filter_kernel   DocIdSetOperator + filter operators.  Per warp: a unit (1-2 x 1024 docs) of every streamed
//     predicate column --cp.async.bulk (TMA) + mbarrier, 2 stages--> smem; lane = 32 consecutive docs: unpack big-endian
//     bit-packed dictIds, evaluate the predicate tree on 32-bit doc masks (one mask word per lane == packed docId
//     bitmap); later leaves of a selective conjunction are tested on the surviving docs only, straight from their forward
//     index; matching docIds reach the global match list in batches through a per-warp shared-memory buffer.
//   pb_agg_kernel      ProjectionOperator + GroupByOperator/AggregationOperator (+ the FILTER clauses of filtered
//     aggregations).  One thread per matching doc: gather group-key / metric dictIds straight from HBM (only the sectors
//     that hold matching rows are touched), dictionary decode, accumulate into the group table with native L2 reductions
//     (RED.ADD.F64 / RED.MIN.S64 / RED.OR.B32).
//
// No tensor cores: the path is integer / gather / atomic bound (BASELINE.json north_star).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PB_NTHREADS 256
#define PB_NWARPS 8
#define PB_CHUNK_DOCS 1024          // docs per warp-chunk (lane owns 32)
#define PB_NSTAGE 2
#define PB_MAX_LEAVES 16
#define PB_MAX_NODES 32
#define PB_MAX_GROUP_BY 16
#define PB_MAX_AGGS 16
#define PB_MAX_SCAN_SLOTS 8
#define PB_MAX_AGG_FILTERS 8         // distinct FILTER(WHERE ...) clauses per query (swim-lanes of FilteredGroupByOperator)
#define PB_MAX_AF_LEAVES 16          // leaves of all FILTER clauses of a segment together
#define PB_MAX_AF_NODES 48
#define PB_SPARSE_MAX 128            // survivors per 1024-doc chunk below which later AND leaves use the restricted scan
#define PB_OUT_CAP 256               // (upper bound; DevQuery::out_cap) matches buffered per warp before one ATOMG reserves their place in the match list
#define PB_CAND_CAP 512              // (upper bound; DevQuery::cand_cap) candidates per warp list (u16 offsets inside the unit); more = extra passes
#define PB_SET_SMEM_BYTES 8192      // dictId-set membership LUTs (one byte per dictId) cached in smem per segment

enum { L_TRUE = 0, L_FALSE = 1, L_DICT_RANGE = 2, L_DICT_SET = 3, L_RAW_RANGE_I = 4, L_RAW_RANGE_F = 5,
       L_RAW_SET = 6, L_BITMAP = 7 };
enum { N_LEAF = 0, N_AND = 1, N_OR = 2, N_NOT = 3 };
enum { T_KEYLESS = 0, T_DENSE = 1, T_HASH = 2 };

#define PB_HASH_EMPTY 0xFFFFFFFFFFFFFFFFull

struct DevLeaf {
  int32_t kind;
  int32_t slot;            // scan slot (tile-staged column) for scan leaves
  int32_t bits;            // dictionary column: bits per element
  int32_t raw_width;       // raw column: 4 or 8
  int32_t data_type;
  int32_t exclusive;
  uint32_t lo, span;       // L_DICT_RANGE: match iff (dictId - lo) < span (unsigned)
  int32_t set_smem_off;    // L_DICT_SET: byte offset of the membership LUT in the smem set cache, -1 = bitset in global
  int32_t set_card;        // dictionary cardinality (LUT length)
  const uint32_t* set_bits;   // L_DICT_SET: bitset over dictIds
  int64_t ilo, ihi;        // L_RAW_RANGE_I inclusive
  double dlo, dhi;         // L_RAW_RANGE_F
  int32_t dlo_incl, dhi_incl;
  const int64_t* raw_set;  // L_RAW_SET
  int32_t n_raw_set;
  int32_t est_permille;    // host estimate of the leaf's selectivity (0..1000), used to order AND chains
  const uint32_t* bitmap;  // L_BITMAP: flat doc bitmap of this segment (bit d&31 of word d>>5)
  // Candidate evaluation (flat AND chains whose earlier leaves leave few survivors): the column of this leaf is NOT
  // streamed through shared memory; the leaf is tested only on the surviving docs, one lane per candidate, reading the
  // forward index where it lies (HBM copy, or the caller's mapped host buffer for cold segments).  The device analogue of
  // SVScanDocIdIterator.applyAnd (CTR/operator/dociditerators/SVScanDocIdIterator.java:115-142).
  int32_t gather;
  uint32_t g_full_words;   // see DevKeyCol::n_full_words
  uint32_t g_tail_word;
  int32_t g_stride_bits;   // bits between consecutive docs' values at gfwd (= bits for a column's own forward index; the row
  int32_t g_bit_off;       // stride and the field offset when the value is read from a row group, see DevKeyCol)
  int32_t pad_l;
  const uint8_t* gfwd;
};

struct DevScanCol {        // a column staged tile-by-tile through smem
  const uint8_t* base;     // first byte of doc 0
  int32_t bits_per_doc;    // bits per element (dict) or 8*raw_width
  int32_t pad;
  uint64_t bytes_total;    // readable bytes from base (16-byte padded)
};

// Gathered columns are read either from their own bit-packed forward index (stride_bits = bits, bit_off = 0) or from a ROW
// GROUP: a second, row-major copy of the columns a query gathers together (group-by keys, aggregation inputs, candidate
// predicate columns), built on the device at first use -- doc d's dictIds packed MSB-first into one row of 64 / 128 / 256
// bits, so that every gather of a matching doc falls into ONE 32-byte DRAM sector instead of one sector per column
// (the aggregation kernel is bound by the DRAM random-access rate, ~50 G sectors/s: profiles/r1_experiments.md).
struct DevKeyCol {         // group-by column (gathered per matching doc)
  const uint8_t* fwd;
  const int32_t* remap;    // local -> global dictId (combined mode), may be null
  int32_t bits;
  int32_t raw_width;       // 0 for dictionary columns
  int32_t data_type;
  int32_t shift;           // T_HASH: bit position of this column in the composite key
  uint64_t mult;           // T_DENSE: mixed-radix multiplier
  uint32_t n_full_words;   // words wholly inside the buffer (0xFFFFFFFF: padded HBM copy, no bound needed)
  uint32_t tail_word;      // in-place host buffer: the trailing partial word, zero-padded (as stored, big-endian)
  int32_t stride_bits;     // bits between consecutive docs' values (bits, or the row stride of a row group)
  int32_t bit_off;         // position of the field inside the row (0 for a column's own forward index)
};

struct DevAggCol {
  const uint8_t* fwd;
  const double* dict_f64;  // dictionary decoded to double
  const int32_t* remap;    // DISTINCTCOUNT in combined mode: local -> global dictId
  int32_t bits;
  int32_t raw_width;
  int32_t data_type;
  uint32_t n_full_words;   // see DevKeyCol
  uint32_t tail_word;
  int32_t stride_bits, bit_off;
  uint32_t pad;
};

struct DevSegQuery {
  int32_t num_docs;
  int32_t n_nodes;
  int32_t n_scan;
  int32_t table;           // result table index
  uint64_t unit_begin;     // global index of this segment's first work unit (U x 1024 docs)
  uint64_t n_units;        // ceil(num_docs / (U * 1024))
  uint64_t doc_base;       // global doc number of this segment's doc 0 (match list numbering)
  int8_t node_kind[PB_MAX_NODES];
  int8_t node_arg[PB_MAX_NODES];
  DevLeaf leaves[PB_MAX_LEAVES];
  DevScanCol scan[PB_MAX_SCAN_SLOTS];
  // ---- everything above is the filter part (copied to shared memory by pb_filter_kernel) ----
  DevKeyCol keys[PB_MAX_GROUP_BY];
  DevAggCol aggs[PB_MAX_AGGS];
  // ---- filtered aggregations: the FILTER(WHERE ...) clauses as postfix programs over leaves that are tested per doc by
  // pb_agg_kernel (clause f = nodes [af_begin[f], af_begin[f+1])); af_docs: docs of this segment that reach the aggregation
  // kernel [0] and that pass clause f [1 + f] (ExecutionStatistics of the swim-lanes) ----
  int32_t n_agg_filters;
  int32_t pad_af;
  int32_t af_begin[PB_MAX_AGG_FILTERS + 1];
  int8_t af_node_kind[PB_MAX_AF_NODES];
  int8_t af_node_arg[PB_MAX_AF_NODES];
  unsigned long long* af_docs;
  DevLeaf af_leaves[PB_MAX_AF_LEAVES];
};
#define PB_SEG_FILTER_BYTES offsetof(DevSegQuery, keys)

struct DevTable {
  int32_t mode;
  int32_t key_words;                 // hash: 1 = 64-bit composite key, 2 = 128-bit (ARRAY_MAP-sized key spaces)
  uint64_t capacity;                 // dense: number of groups; hash: slots (power of two)
  unsigned long long* hkeys;         // hash: slot keys (PB_HASH_EMPTY = free)
  unsigned long long* rowcnt;        // rows per slot
  double* sum[PB_MAX_AGGS];
  long long* mm[PB_MAX_AGGS];        // order-preserving int64 encoding of the double min / max
  unsigned long long* fcnt[PB_MAX_AGGS];   // COUNT / AVG with a FILTER clause: their own row count (others use rowcnt)
  uint32_t* dc_bits[PB_MAX_AGGS];    // DISTINCTCOUNT: per-slot bitset over (global) dictIds
  uint64_t dc_words[PB_MAX_AGGS];
  // DISTINCTCOUNT on a raw column (the reference keeps a value set per group: BaseDistinctAggregateAggregationFunction.java:
  // 157-226): ONE open-addressing set of (slot, value bits) pairs for the whole table, 16-byte entries claimed with CAS.128;
  // dcnt[slot] = distinct values of the slot, counted from the set at hand-back
  unsigned long long* dset[PB_MAX_AGGS];
  uint64_t dset_mask[PB_MAX_AGGS];
  unsigned long long* dcnt[PB_MAX_AGGS];
  unsigned int* num_groups;          // hash: groups created so far
  unsigned int* limit_reached;
  unsigned int* any_limit;           // query-wide: some hash table of this launch refused a key (drives the repair pass)
  unsigned long long* docs_matched;  // numDocsScanned
  // dense table whose key space exceeds numGroupsLimit (the reference's IntMapBasedHolder, first come first served in doc
  // order: DictionaryBasedGroupKeyGenerator.java:1023-1058): first_doc[slot] = smallest doc that produced the group; the
  // hand-back keeps the numGroupsLimit groups that appeared first -- exactly the groups the reference would have created
  uint32_t* first_doc;
  uint32_t num_groups_limit;
  uint32_t limit_active;             // 0: the table can never reach numGroupsLimit (limit >= docs), inserts need no ticket
};

struct DevQuery {
  int32_t n_segs;
  int32_t n_group_by;
  int32_t n_aggs;
  int32_t table_mode;
  int32_t agg_op[PB_MAX_AGGS];
  int32_t agg_filter_of[PB_MAX_AGGS];    // FILTER clause of each aggregation (-1 = none)
  int32_t n_agg_filters;
  int32_t pad_f;
  int32_t slot_off[PB_MAX_SCAN_SLOTS];   // byte offset of each scan slot inside a stage
  int32_t stage_bytes;                   // bytes per warp stage (one 1024-doc chunk of every scan slot)
  int32_t set_cache_bytes;               // shared-memory bytes reserved for IN-set membership LUTs
  int32_t use_tma;
  int32_t generic;                       // 1 = width-generic predicate path only
  uint64_t n_units;
  uint64_t n_docs_total;
  int32_t match_all;                     // no filter: pb_agg_kernel walks every doc, no match list
  int32_t agg_counts_docs;               // some segment has residual leaves (DevRowLeaf): the match list holds candidates and
                                         // pb_agg_rows_kernel, not the filter kernel, counts docs_matched
  int32_t sparse_max;                    // survivors per 1024 docs below which later AND leaves use the restricted scan
  int32_t cand_bytes;                    // shared memory for the per-warp candidate lists (0: no leaf runs on candidates)
  uint64_t unit_lo;                      // this launch covers work units [unit_lo, unit_lo + n_units) (a wave of segments)
  int32_t phase;                         // pb_agg_kernel: 0 = normal; 2 = repair pass of a hash table that hit numGroupsLimit (see pb_hash_slot)
  int32_t st_slots;                      // pb_agg_smem_kernel: slots of the CTA-private dense table (= table capacity), 0 = not used
  int32_t st_replicas;                   //   replicas of it per CTA (power of two)
  int32_t out_cap, cand_cap;             // per-warp output buffer / candidate list entries (smaller caps let a fourth CTA fit an SM)
  uint64_t st_min_docs;                  //   matches below which the kernel updates the global table directly (merging 148 private tables costs more)
  uint32_t* match_list;                  // global doc numbers of the docs that pass the filter
  unsigned long long* match_count;
  const unsigned int* any_limit;         // see DevTable::any_limit
  const DevSegQuery* segs;
  DevTable* tables;
};

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pb_bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

// order-preserving int64 encoding of a double (signed compare == double compare)
__device__ __forceinline__ long long pb_enc_f64(double v) {
  long long b = __double_as_longlong(v);
  return b >= 0 ? b : (b ^ 0x7fffffffffffffffLL);
}
__host__ __device__ __forceinline__ double pb_dec_f64(long long e) {
  long long b = e >= 0 ? e : (e ^ 0x7fffffffffffffffLL);
#ifdef __CUDA_ARCH__
  return __longlong_as_double(b);
#else
  double d; memcpy(&d, &b, 8); return d;
#endif
}

// dictId of `doc` from a big-endian MSB-first bitstream in global memory
// (FixedBitSVForwardIndexReaderV2.readDictIds, SEGL/segment/index/readers/forward/FixedBitSVForwardIndexReaderV2.java:65-99;
//  bit layout SEGL/io/util/PinotDataBitSet.java:80-102).  The buffer is 4-byte aligned and padded by >= 8 bytes.
__device__ __forceinline__ uint32_t pb_unpack_at(const uint8_t* __restrict__ fwd, uint32_t doc, int bits) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(fwd);
  unsigned long long bit = (unsigned long long)doc * (unsigned)bits;
  unsigned long long wi = bit >> 5;
  uint32_t s = (uint32_t)bit & 31u;
  uint32_t hi = pb_bswap32(__ldg(w + wi));
  uint32_t lo = pb_bswap32(__ldg(w + wi + 1));
  return __funnelshift_l(lo, hi, s) >> (32 - bits);
}

// Same, for a gathered column that may be read IN PLACE from the caller's page-locked host buffer (PB_Q_GATHER_IN_PLACE):
// that buffer has no padding, so words past its last whole word come from the descriptor instead of memory.
__device__ __forceinline__ uint32_t pb_unpack_at_bounded(const uint8_t* __restrict__ fwd, uint32_t doc, int bits, uint32_t n_full, uint32_t tail,
                                                         int stride_bits, int bit_off) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(fwd);
  unsigned long long bit = (unsigned long long)doc * (unsigned)stride_bits + (unsigned)bit_off;
  unsigned long long wi = bit >> 5;
  uint32_t s = (uint32_t)bit & 31u;
  uint32_t hi = tail, lo = tail;
  if (wi < n_full) hi = __ldg(w + wi);
  if (wi + 1 < n_full) lo = __ldg(w + wi + 1);
  return __funnelshift_l(pb_bswap32(lo), pb_bswap32(hi), s) >> (32 - bits);
}

// raw PASS_THROUGH forward index value (FixedByteChunkSVForwardIndexReader.java:53-61): big-endian
// stride_bits / bit_off: a column's own raw forward index has stride 8 * width and offset 0; a DECODED VALUE field of a row
// group (see DevKeyCol) has the row stride and its (32-bit aligned) offset inside the row
__device__ __forceinline__ long long pb_raw_i64(const uint8_t* __restrict__ fwd, uint32_t doc, int width, int data_type, int stride_bits, int bit_off) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(fwd) + (((unsigned long long)doc * (unsigned)stride_bits + (unsigned)bit_off) >> 5);
  if (width == 4) return (long long)(int32_t)pb_bswap32(__ldg(w));
  uint32_t hi = pb_bswap32(__ldg(w)), lo = pb_bswap32(__ldg(w + 1));
  return (long long)(((unsigned long long)hi << 32) | lo);
}
__device__ __forceinline__ double pb_raw_f64(const uint8_t* __restrict__ fwd, uint32_t doc, int width, int data_type, int stride_bits, int bit_off) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(fwd) + (((unsigned long long)doc * (unsigned)stride_bits + (unsigned)bit_off) >> 5);
  if (width == 4) {
    uint32_t u = pb_bswap32(__ldg(w));
    return data_type == 2 ? (double)__uint_as_float(u) : (double)(int32_t)u;
  }
  uint32_t hi = pb_bswap32(__ldg(w)), lo = pb_bswap32(__ldg(w + 1));
  unsigned long long u = ((unsigned long long)hi << 32) | lo;
  return data_type == 3 ? __longlong_as_double((long long)u) : (double)(long long)u;
}


// ---- global-memory reductions (SASS REDG.*): the table pointers are loaded from descriptors, so the
// compiler cannot prove the address space; state it explicitly instead of going through generic ATOM + isspacep.
__device__ __forceinline__ void pb_red_add_f64(double* p, double v) { asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v)); }
__device__ __forceinline__ void pb_red_add_u64(unsigned long long* p, unsigned long long v) { asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v)); }
__device__ __forceinline__ void pb_red_add_u32(unsigned int* p, unsigned int v) { asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v)); }
__device__ __forceinline__ void pb_red_min_s64(long long* p, long long v) { asm volatile("red.global.min.s64 [%0], %1;" ::"l"(p), "l"(v)); }
__device__ __forceinline__ void pb_red_max_s64(long long* p, long long v) { asm volatile("red.global.max.s64 [%0], %1;" ::"l"(p), "l"(v)); }
__device__ __forceinline__ void pb_red_or_b32(uint32_t* p, uint32_t v) { asm volatile("red.global.or.b32 [%0], %1;" ::"l"(p), "r"(v)); }
__device__ __forceinline__ unsigned long long pb_atom_cas_u64(unsigned long long* p, unsigned long long cmp, unsigned long long val) {
  unsigned long long old;
  asm volatile("atom.global.cas.b64 %0, [%1], %2, %3;" : "=l"(old) : "l"(p), "l"(cmp), "l"(val) : "memory");
  return old;
}
__device__ __forceinline__ unsigned int pb_atom_add_u32(unsigned int* p, unsigned int v) {
  unsigned int old;
  asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ unsigned long long pb_ld_volatile_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned int pb_ld_volatile_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---- mbarrier / TMA bulk copy (cp.async.bulk -> SASS UBLKCP) ----
__device__ __forceinline__ uint32_t pb_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void pb_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pb_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void pb_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pb_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t pb_mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(pb_smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void pb_mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!pb_mbar_try_wait(bar, parity)) {}
}
// streaming variant: the scanned columns are read once (evict-first), the gathered sectors and tables stay in L2
__device__ __forceinline__ uint64_t pb_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void pb_tma_load_1d_hint(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                   pb_smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(pb_smem_u32(bar)), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void pb_tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   pb_smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(pb_smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------------------------------------
// predicate evaluation on one 1024-doc chunk; every variant returns THIS LANE's 32-bit mask for docs
// [chunk_doc0 + 32*lane, +32)   (PredicateEvaluator.applySV semantics, CTR/operator/filter/predicate/*)
// ------------------------------------------------------------------------------------------------
// Each functor sees the value TOP-ALIGNED in 32 bits (vt = dictId << (32-W) | garbage below the field) so a
// range test needs no masking; returns 0/1.
struct PredRange {      // SortedDictionaryBasedRangePredicateEvaluator.applySV: start <= dictId < end
  uint32_t lo, span;
  template <int W> __device__ __forceinline__ uint32_t test(uint32_t vt) const {
    return ((vt - (lo << (32 - W))) < (span << (32 - W))) ? 1u : 0u;
  }
  __device__ __forceinline__ uint32_t operator()(uint32_t v) const { return (v - lo) < span ? 1u : 0u; }
};
struct PredLut8 {       // IN / NOT_IN / EQ / NEQ: one membership byte per dictId in shared memory, exclusive flag folded in.
                        // (A bitset is conflict-free but costs ~3 more ALU instructions per value; the kernel is issue-bound,
                        // the shared-memory pipe is only ~25 % busy: profiles/r1_experiments.md.)
  const uint8_t* lut;
  template <int W> __device__ __forceinline__ uint32_t test(uint32_t vt) const { return lut[vt >> (32 - W)]; }
  __device__ __forceinline__ uint32_t operator()(uint32_t v) const { return lut[v]; }
};
struct PredBits {       // same, large dictionaries: bitset in global memory (L1-resident)
  const uint32_t* bits;
  uint32_t excl;
  template <int W> __device__ __forceinline__ uint32_t test(uint32_t vt) const { return (*this)(vt >> (32 - W)); }
  __device__ __forceinline__ uint32_t operator()(uint32_t v) const { return (__funnelshift_r(__ldg(bits + (v >> 5)), 0u, v) & 1u) ^ excl; }
};

// width-generic path: lane <-> doc, 32 steps, ballot; conflict-free smem reads
template <class Pred>
__device__ __forceinline__ uint32_t pb_eval_dict_generic(const uint32_t* __restrict__ p, int bits, const Pred& pred, int lane) {
  uint32_t mine = 0;
#pragma unroll 4
  for (int k = 0; k < 32; k++) {
    uint32_t idx = (uint32_t)(k * 32 + lane);
    uint32_t bit = idx * (uint32_t)bits;
    uint32_t wi = bit >> 5, s = bit & 31u;
    uint32_t hi = pb_bswap32(p[wi]), lo = pb_bswap32(p[wi + 1]);
    uint32_t v = __funnelshift_l(lo, hi, s) >> (32 - bits);
    uint32_t b = __ballot_sync(0xffffffffu, pred(v) != 0);
    if (k == lane) mine = b;
  }
  return mine;
}

// width-specialised path: lane owns 32 consecutive docs == exactly W consecutive 32-bit words.
// All shifts are compile-time constants (the GPU analogue of FixedBitIntReader's per-width read32 classes,
// SEGL/io/reader/impl/FixedBitIntReader.java:121-146).  The mask is built MSB-first by shift-accumulate.
template <int W, class Pred>
__device__ __forceinline__ uint32_t pb_eval_dict_w(const uint32_t* __restrict__ p, const Pred& pred, int lane) {
  uint32_t w[W + 1];
  const uint32_t* q = p + lane * W;
#pragma unroll
  for (int k = 0; k < W; k++) w[k] = pb_bswap32(q[k]);
  w[W] = 0;
  // four independent shift-accumulate chains (8 docs each) instead of one 32-deep dependency chain
  uint32_t m[4] = {0, 0, 0, 0};
#pragma unroll
  for (int j = 31; j >= 0; j--) {
    const int bit = j * W;
    const int k = bit >> 5, s = bit & 31;
    const uint32_t vt = (s == 0) ? w[k] : __funnelshift_l(w[k + 1], w[k], s);   // value in the top W bits
    m[j >> 3] = m[j >> 3] * 2 + pred.template test<W>(vt);
  }
  return (m[3] << 24) | (m[2] << 16) | (m[1] << 8) | m[0];
}

// restricted scan: only the docs still set in `mask` are decoded and tested (the device analogue of
// SVScanDocIdIterator.applyAnd over the surviving docIds, CTR/operator/dociditerators/SVScanDocIdIterator.java:115-142)
template <class Pred>
__device__ __forceinline__ uint32_t pb_eval_dict_sparse(const uint32_t* __restrict__ p, int bits, const Pred& pred, int lane, uint32_t mask) {
  const uint32_t* q = p + lane * bits;
  uint32_t rem = mask;
  while (rem) {
    const int j = __ffs(rem) - 1;
    rem &= rem - 1;
    const uint32_t bit = (uint32_t)j * (uint32_t)bits;
    const uint32_t k = bit >> 5, s = bit & 31u;
    const uint32_t hi = pb_bswap32(q[k]), lo = pb_bswap32(q[k + 1]);
    const uint32_t v = __funnelshift_l(lo, hi, s) >> (32 - bits);
    if (!pred(v)) mask &= ~(1u << j);
  }
  return mask;
}

__device__ __forceinline__ bool pb_fast_width(int bits) { return bits < 32 && (bits & 7) != 0; }

// evaluates nu (<= 2) consecutive 1024-doc chunks with one dispatch: out[u] = this lane's mask of sub-chunk u
template <class Pred>
__device__ __noinline__ void pb_eval_dict_fast(const uint32_t* __restrict__ p, int bits, const Pred& pred, int lane, int nu, uint32_t* out) {
  switch (bits) {
#define PB_CASE(W) case W: for (int u = 0; u < nu; u++) out[u] = pb_eval_dict_w<W, Pred>(p + u * 32 * W, pred, lane); return;
    PB_CASE(1) PB_CASE(2) PB_CASE(3) PB_CASE(4) PB_CASE(5) PB_CASE(6) PB_CASE(7)
    PB_CASE(9) PB_CASE(10) PB_CASE(11) PB_CASE(12) PB_CASE(13) PB_CASE(14) PB_CASE(15)
    PB_CASE(17) PB_CASE(18) PB_CASE(19) PB_CASE(20) PB_CASE(21) PB_CASE(22) PB_CASE(23)
    PB_CASE(25) PB_CASE(26) PB_CASE(27) PB_CASE(28) PB_CASE(29) PB_CASE(30) PB_CASE(31)
#undef PB_CASE
    default: for (int u = 0; u < nu; u++) out[u] = 0; return;
  }
}

template <class Pred>
__device__ __forceinline__ void pb_eval_dict(const uint32_t* __restrict__ p, int bits, const Pred& pred, int lane, bool generic, int nu, uint32_t* out) {
  if (!generic && pb_fast_width(bits)) { pb_eval_dict_fast<Pred>(p, bits, pred, lane, nu, out); return; }
  for (int u = 0; u < nu; u++) out[u] = pb_eval_dict_generic<Pred>(p + u * 32 * bits, bits, pred, lane);
}

// raw fixed-width column chunk in smem (big-endian values), lane <-> doc + ballot
static __device__ __noinline__ uint32_t pb_eval_raw(const uint32_t* __restrict__ p, const DevLeaf& lf, int lane) {
  uint32_t mine = 0;
  for (int k = 0; k < 32; k++) {
    uint32_t idx = (uint32_t)(k * 32 + lane);
    bool ok;
    if (lf.raw_width == 4) {
      uint32_t u = pb_bswap32(p[idx]);
      if (lf.data_type == 2) {   // FLOAT
        double v = (double)__uint_as_float(u);
        if (lf.kind == L_RAW_RANGE_F) ok = (lf.dlo_incl ? v >= lf.dlo : v > lf.dlo) && (lf.dhi_incl ? v <= lf.dhi : v < lf.dhi);
        else { bool in = false; long long vb = __double_as_longlong(v); for (int i = 0; i < lf.n_raw_set; i++) in |= (lf.raw_set[i] == vb); ok = in != (bool)lf.exclusive; }
      } else {                   // INT
        long long v = (long long)(int32_t)u;
        if (lf.kind == L_RAW_RANGE_I) ok = v >= lf.ilo && v <= lf.ihi;
        else { bool in = false; for (int i = 0; i < lf.n_raw_set; i++) in |= (lf.raw_set[i] == v); ok = in != (bool)lf.exclusive; }
      }
    } else {
      unsigned long long u = ((unsigned long long)pb_bswap32(p[2 * idx]) << 32) | pb_bswap32(p[2 * idx + 1]);
      if (lf.data_type == 3) {   // DOUBLE
        double v = __longlong_as_double((long long)u);
        if (lf.kind == L_RAW_RANGE_F) ok = (lf.dlo_incl ? v >= lf.dlo : v > lf.dlo) && (lf.dhi_incl ? v <= lf.dhi : v < lf.dhi);
        else { bool in = false; for (int i = 0; i < lf.n_raw_set; i++) in |= (lf.raw_set[i] == (long long)u); ok = in != (bool)lf.exclusive; }
      } else {                   // LONG
        long long v = (long long)u;
        if (lf.kind == L_RAW_RANGE_I) ok = v >= lf.ilo && v <= lf.ihi;
        else { bool in = false; for (int i = 0; i < lf.n_raw_set; i++) in |= (lf.raw_set[i] == v); ok = in != (bool)lf.exclusive; }
      }
    }
    uint32_t b = __ballot_sync(0xffffffffu, ok);
    if (k == lane) mine = b;
  }
  return mine;
}

// one doc against one scan leaf, reading the forward index in place (candidate evaluation, see DevLeaf::gather)
__device__ __forceinline__ bool pb_leaf_test_doc(const DevLeaf& lf, const uint8_t* __restrict__ set_cache, uint32_t doc) {
  switch (lf.kind) {
    case L_TRUE: return true;
    case L_FALSE: return false;
    case L_DICT_RANGE: {
      const uint32_t id = pb_unpack_at_bounded(lf.gfwd, doc, lf.bits, lf.g_full_words, lf.g_tail_word, lf.g_stride_bits, lf.g_bit_off);
      return (id - lf.lo) < lf.span;
    }
    case L_DICT_SET: {
      const uint32_t id = pb_unpack_at_bounded(lf.gfwd, doc, lf.bits, lf.g_full_words, lf.g_tail_word, lf.g_stride_bits, lf.g_bit_off);
      if (lf.set_smem_off >= 0) return set_cache[lf.set_smem_off + id] != 0;         // exclusive flag folded in
      return (((__ldg(lf.set_bits + (id >> 5)) >> (id & 31)) & 1u) ^ (uint32_t)lf.exclusive) != 0;
    }
    case L_BITMAP: return (((__ldg(lf.bitmap + (doc >> 5)) >> (doc & 31)) & 1u) ^ (uint32_t)lf.exclusive) != 0;
    case L_RAW_RANGE_I: { const long long v = pb_raw_i64(lf.gfwd, doc, lf.raw_width, lf.data_type, lf.g_stride_bits, lf.g_bit_off); return v >= lf.ilo && v <= lf.ihi; }
    case L_RAW_RANGE_F: {
      const double v = pb_raw_f64(lf.gfwd, doc, lf.raw_width, lf.data_type, lf.g_stride_bits, lf.g_bit_off);
      return (lf.dlo_incl ? v >= lf.dlo : v > lf.dlo) && (lf.dhi_incl ? v <= lf.dhi : v < lf.dhi);
    }
    case L_RAW_SET: {
      long long vb;
      if (lf.data_type == 2 || lf.data_type == 3) vb = __double_as_longlong(pb_raw_f64(lf.gfwd, doc, lf.raw_width, lf.data_type, lf.g_stride_bits, lf.g_bit_off));
      else vb = pb_raw_i64(lf.gfwd, doc, lf.raw_width, lf.data_type, lf.g_stride_bits, lf.g_bit_off);
      bool in = false;
      for (int i = 0; i < lf.n_raw_set; i++) in |= (lf.raw_set[i] == vb);
      return in != (bool)lf.exclusive;
    }
    default: return false;
  }
}

// ------------------------------------------------------------------------------------------------
// group table update for one matching doc
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t pb_hash64(uint64_t k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return k;
}

// ---- numGroupsLimit (DictionaryBasedGroupKeyGenerator.java:1033-1035: a NEW key past the limit gets INVALID_ID and its
// rows are dropped; existing keys keep aggregating).  A thread may insert only while it holds a ticket, taken from
// num_groups with a returning atomic BEFORE the slot is claimed (the check-then-insert of round 1 let every resident thread
// pass the check at once and could fill the table, after which absent keys probed forever).  Tickets are never handed
// back: once one request has been refused every later one is refused too, so a key can never be created after some of its
// rows were dropped (no partially aggregated group) and the table never holds more than `limit` keys; a claim lost to a
// concurrent insert of the same slot wastes its ticket, so a limited result may hold a few groups fewer than the limit.
// Lanes of a warp that need a ticket at the same time share one atomic.  Probing is bounded by the capacity.
// One anomaly is left to a REPAIR PASS: a row can be refused while another thread that already holds a ticket is about to
// create the very same key, which would leave that group short of the refused row.  When (and only when) some key was
// refused, the aggregates are zeroed again (the keys stay) and the matches are aggregated a second time in lookup-only mode
// (DevQuery::phase = 2): every row of a key that made it into the table counts, every other row is dropped -- exactly the
// reference's "existing groups keep aggregating, new keys are ignored". ----
__device__ __forceinline__ bool pb_group_ticket(const DevTable& t) {
  if (!t.limit_active) return true;                      // groups <= docs <= limit: cannot be reached, nothing to count
  const unsigned m = __activemask();
  const int leader = __ffs(m) - 1, lane = (int)(threadIdx.x & 31);
  const unsigned rank = __popc(m & ((1u << lane) - 1u)), need = __popc(m);
  unsigned base = 0;
  if (lane == leader) base = pb_atom_add_u32(t.num_groups, need);
  base = __shfl_sync(m, base, leader);
  if (base + rank < t.num_groups_limit) return true;
  pb_red_add_u32(t.limit_reached, 1u);
  if (t.any_limit) pb_red_add_u32(t.any_limit, 1u);
  return false;
}
__device__ __forceinline__ void pb_group_ticket_return(const DevTable&) {}

// returns slot, or ~0ull when the key is new and numGroupsLimit is reached
__device__ __forceinline__ uint64_t pb_hash_slot(const DevTable& t, uint64_t key, bool insert = true) {
  if (key == PB_HASH_EMPTY) return t.capacity;          // reserved extra slot for the sentinel value itself
  uint64_t mask = t.capacity - 1;
  uint64_t s = pb_hash64(key) & mask;
  for (uint64_t probes = 0; probes <= mask; probes++) {
    unsigned long long cur = pb_ld_volatile_u64(&t.hkeys[s]);
    if (cur == key) return s;
    if (cur == PB_HASH_EMPTY) {
      // the key is not in the table (linear probing never skips an empty slot): inserting needs a ticket
      if (!insert || !pb_group_ticket(t)) return ~0ull;
      unsigned long long old = pb_atom_cas_u64(&t.hkeys[s], PB_HASH_EMPTY, (unsigned long long)key);
      if (old == PB_HASH_EMPTY) return s;
      pb_group_ticket_return(t);                         // somebody else claimed the slot first
      if (old == key) return s;
    }
    s = (s + 1) & mask;
  }
  pb_red_add_u32(t.limit_reached, 1u);                   // table full (cannot happen while capacity >= 2 x limit): drop the row
  return ~0ull;
}

// 128-bit composite keys (more than 64 bits of dictIds: the reference's ArrayMapBasedHolder,
// DictionaryBasedGroupKeyGenerator.java:809-885): slots are 16-byte pairs claimed with ATOMG.CAS.128
__device__ __forceinline__ void pb_atom_cas_u128(unsigned long long* p, unsigned long long clo, unsigned long long chi, unsigned long long vlo,
                                                 unsigned long long vhi, unsigned long long& olo, unsigned long long& ohi) {
  asm volatile("{\n.reg .b128 c, v, o;\nmov.b128 c, {%2, %3};\nmov.b128 v, {%4, %5};\natom.global.cas.b128 o, [%6], c, v;\nmov.b128 {%0, %1}, o;\n}\n"
               : "=l"(olo), "=l"(ohi) : "l"(clo), "l"(chi), "l"(vlo), "l"(vhi), "l"(p) : "memory");
}
__device__ __forceinline__ uint64_t pb_hash_slot2(const DevTable& t, uint64_t lo, uint64_t hi, bool insert = true) {
  if (lo == PB_HASH_EMPTY && hi == PB_HASH_EMPTY) return t.capacity;     // reserved slot for the sentinel pattern itself
  const uint64_t mask = t.capacity - 1;
  uint64_t s = pb_hash64(lo ^ pb_hash64(hi)) & mask;
  for (uint64_t probes = 0; probes <= mask; probes++) {
    unsigned long long clo, chi;   // one 16-byte transaction, so a concurrent CAS.128 is seen whole or not at all
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(clo), "=l"(chi) : "l"(&t.hkeys[2 * s]));
    if (clo == lo && chi == hi) return s;
    if (clo == PB_HASH_EMPTY && chi == PB_HASH_EMPTY) {
      if (!insert || !pb_group_ticket(t)) return ~0ull;
      unsigned long long olo, ohi;
      pb_atom_cas_u128(&t.hkeys[2 * s], PB_HASH_EMPTY, PB_HASH_EMPTY, lo, hi, olo, ohi);
      if (olo == PB_HASH_EMPTY && ohi == PB_HASH_EMPTY) return s;
      pb_group_ticket_return(t);
      if (olo == lo && ohi == hi) return s;
    }
    s = (s + 1) & mask;
  }
  pb_red_add_u32(t.limit_reached, 1u);
  return ~0ull;
}

// keyless accumulators live in shared memory, one private cell per thread (no atomics)
struct KeylessAcc {
  double* sum;               // [n_aggs][PB_NTHREADS]
  long long* mm;             // [n_aggs][PB_NTHREADS]
  unsigned long long* cnt;   // [n_aggs][PB_NTHREADS]: row counts of COUNT / AVG with a FILTER clause (null without clauses)
};

// FILTER(WHERE ...) clauses of the query against one doc: bit f of the result = clause f passes
// (the swim-lane filters of FilteredGroupByOperator.java:108-159, evaluated per doc instead of per lane)
__device__ __forceinline__ uint32_t pb_agg_filter_bits(const DevSegQuery& sq, uint32_t doc) {
  uint32_t bits = 0;
  for (int f = 0; f < sq.n_agg_filters; f++) {
    uint32_t stack = 0;       // boolean stack, top = bit 0
    for (int n = sq.af_begin[f]; n < sq.af_begin[f + 1]; n++) {
      const int kind = sq.af_node_kind[n], arg = sq.af_node_arg[n];
      if (kind == N_LEAF) stack = (stack << 1) | (pb_leaf_test_doc(sq.af_leaves[arg], nullptr, doc) ? 1u : 0u);
      else if (kind == N_NOT) stack ^= 1u;
      else {
        const uint32_t m = (1u << arg) - 1u, top = stack & m;
        const uint32_t r = kind == N_AND ? (top == m ? 1u : 0u) : (top != 0u ? 1u : 0u);
        stack = ((stack >> arg) << 1) | r;
      }
    }
    if (sq.af_begin[f + 1] == sq.af_begin[f] || (stack & 1u)) bits |= 1u << f;      // an empty program matches all
  }
  return bits;
}

__device__ __forceinline__ uint64_t pb_key_field(const DevKeyCol& kc, uint32_t doc, bool multi) {
  if (kc.raw_width) {
    uint64_t v;
    if (kc.data_type == 2 || kc.data_type == 3) v = (uint64_t)__double_as_longlong(pb_raw_f64(kc.fwd, doc, kc.raw_width, kc.data_type, kc.stride_bits, kc.bit_off));
    else v = (uint64_t)pb_raw_i64(kc.fwd, doc, kc.raw_width, kc.data_type, kc.stride_bits, kc.bit_off);
    return (kc.raw_width == 4 && multi) ? (v & 0xffffffffull) : v;
  }
  uint32_t id = pb_unpack_at_bounded(kc.fwd, doc, kc.bits, kc.n_full_words, kc.tail_word, kc.stride_bits, kc.bit_off);
  if (kc.remap) id = (uint32_t)__ldg(kc.remap + id);
  return id;
}

// value of aggregation column a for `doc`: BlockValSet.getDoubleValuesSV (dictionary decode or raw read, widened
// to double); for DISTINCTCOUNT the (global) dictId, returned through the same 64-bit channel
__device__ __forceinline__ double pb_agg_input(const DevAggCol& ac, int op, uint32_t doc) {
  if (op == 5 && ac.raw_width) {       // raw column: the value itself, as bits (NaNs canonical, like Double.doubleToLongBits)
    if (ac.data_type == 2 || ac.data_type == 3) { const double d = pb_raw_f64(ac.fwd, doc, ac.raw_width, ac.data_type, ac.stride_bits, ac.bit_off); return d == d ? d : __longlong_as_double(0x7ff8000000000000LL); }
    return __longlong_as_double(pb_raw_i64(ac.fwd, doc, ac.raw_width, ac.data_type, ac.stride_bits, ac.bit_off));
  }
  if (op == 5) {
    uint32_t id = pb_unpack_at_bounded(ac.fwd, doc, ac.bits, ac.n_full_words, ac.tail_word, ac.stride_bits, ac.bit_off);
    if (ac.remap) id = (uint32_t)__ldg(ac.remap + id);
    return __longlong_as_double((long long)id);
  }
  return ac.raw_width ? pb_raw_f64(ac.fwd, doc, ac.raw_width, ac.data_type, ac.stride_bits, ac.bit_off)
                      : __ldg(ac.dict_f64 + pb_unpack_at_bounded(ac.fwd, doc, ac.bits, ac.n_full_words, ac.tail_word, ac.stride_bits, ac.bit_off));
}

// (slot, value) into the table-wide distinct set of aggregation a
__device__ __forceinline__ void pb_dset_insert(const DevTable& t, int a, uint64_t slot, unsigned long long v) {
  const uint64_t mask = t.dset_mask[a];
  unsigned long long* keys = t.dset[a];
  uint64_t s = pb_hash64(slot * 0x9e3779b97f4a7c15ull ^ pb_hash64(v)) & mask;
  for (uint64_t probes = 0; probes <= mask; probes++) {
    unsigned long long clo, chi;
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(clo), "=l"(chi) : "l"(&keys[2 * s]));
    if (clo == slot && chi == v) return;
    if (clo == PB_HASH_EMPTY && chi == PB_HASH_EMPTY) {
      unsigned long long olo, ohi;
      pb_atom_cas_u128(&keys[2 * s], PB_HASH_EMPTY, PB_HASH_EMPTY, slot, v, olo, ohi);
      if ((olo == PB_HASH_EMPTY && ohi == PB_HASH_EMPTY) || (olo == slot && ohi == v)) return;
    }
    s = (s + 1) & mask;
  }
}

// ---- phase 1 of a matching doc: every gather is issued before anything is reduced, four independent chains at a
// time (index clamping instead of branches keeps the loads unconditional, so they overlap).  slot = dense table index,
// or the 64 / 128-bit composite key of a hash table. ----
__device__ __forceinline__ void pb_gather_doc(const DevQuery& Q, const DevSegQuery& sq, uint32_t doc, uint64_t& slot, uint64_t& slot_hi, double* vals) {
  const int nG = Q.n_group_by, nA = Q.n_aggs;
  slot = 0; slot_hi = 0;
  if (Q.table_mode != T_KEYLESS) {
    const bool dense = Q.table_mode == T_DENSE;
    const bool multi = nG > 1;
    for (int j = 0; j < nG; j += 4) {
      uint64_t f[4];
#pragma unroll
      for (int k = 0; k < 4; k++) f[k] = pb_key_field(sq.keys[min(j + k, nG - 1)], doc, multi);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (j + k < nG) {
          const DevKeyCol& kc = sq.keys[j + k];
          if (dense) slot += f[k] * kc.mult;
          else if (kc.shift < 64) { slot |= f[k] << kc.shift; if (kc.shift) slot_hi |= f[k] >> (64 - kc.shift); }
          else slot_hi |= f[k] << (kc.shift - 64);
        }
      }
    }
  }
  for (int a = 0; a < nA; a += 4) {
    double v[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int aa = min(a + k, nA - 1);
      const int op = Q.agg_op[aa];
      v[k] = op == 0 ? 0.0 : pb_agg_input(sq.aggs[aa], op, doc);
    }
#pragma unroll
    for (int k = 0; k < 4; k++) if (a + k < nA) vals[a + k] = v[k];
  }
}

__device__ __forceinline__ void pb_accumulate(const DevQuery& Q, const DevSegQuery& sq, const DevTable& t, uint32_t doc,
                                              const KeylessAcc& ka, unsigned long long& keyless_rows, uint32_t fpass) {
  const int nA = Q.n_aggs;
  uint64_t slot, slot_hi;
  double vals[PB_MAX_AGGS];
  pb_gather_doc(Q, sq, doc, slot, slot_hi, vals);

  // ---- phase 2: table update ----
  if (Q.table_mode == T_HASH) {
    const bool insert = Q.phase != 2;
    slot = t.key_words == 2 ? pb_hash_slot2(t, slot, slot_hi, insert) : pb_hash_slot(t, slot, insert);
    if (slot == ~0ull) return;
  }
  if (Q.table_mode == T_KEYLESS) keyless_rows++;
  else pb_red_add_u64(&t.rowcnt[slot], 1ull);
  if (t.first_doc) asm volatile("red.global.min.u32 [%0], %1;" ::"l"(t.first_doc + slot), "r"(doc));

  for (int a = 0; a < nA; a++) {
    const int op = Q.agg_op[a];
    const int fo = Q.agg_filter_of[a];
    if (fo >= 0) {                               // FILTER clause: the function only sees docs that pass it
      if (!((fpass >> fo) & 1u)) continue;
      if (t.fcnt[a]) {                           // its own row count (COUNT value / AVG denominator; every function with PB_Q_NULL_HANDLING)
        if (Q.table_mode == T_KEYLESS) ka.cnt[a * PB_NTHREADS + threadIdx.x]++;
        else pb_red_add_u64(&t.fcnt[a][slot], 1ull);
      }
    }
    if (op == 0) continue;                       // COUNT(*): the row counter
    const double v = vals[a];
    if (op == 5) {                               // DISTINCTCOUNT: dictionary column -> bitset over dictIds; raw column -> value set
      if (t.dset[a]) { pb_dset_insert(t, a, slot, (unsigned long long)__double_as_longlong(v)); continue; }
      uint32_t id = (uint32_t)__double_as_longlong(v);
      pb_red_or_b32(&t.dc_bits[a][slot * t.dc_words[a] + (id >> 5)], 1u << (id & 31));
      continue;
    }
    if (Q.table_mode == T_KEYLESS) {
      const int tid = threadIdx.x;
      if (op == 1 || op == 4) ka.sum[a * PB_NTHREADS + tid] += v;
      else if (v == v) {
        long long e = pb_enc_f64(v);
        long long c = ka.mm[a * PB_NTHREADS + tid];
        if (op == 2 ? e < c : e > c) ka.mm[a * PB_NTHREADS + tid] = e;
      }
    } else {
      if (op == 1 || op == 4) pb_red_add_f64(&t.sum[a][slot], v);            // REDG.E.ADD.F64
      else if (v == v) {                                                      // NaN never replaces (strict compare)
        // MAX is kept as MIN of the bit-complement (one init value for all).  Most docs do not improve the extreme: a plain
        // (possibly stale: the RED still decides) read filters them out before they reach the L2 atomic units
        const long long e = op == 2 ? pb_enc_f64(v) : ~pb_enc_f64(v);
        if (e < (long long)pb_ld_volatile_u64(reinterpret_cast<const unsigned long long*>(&t.mm[a][slot]))) pb_red_min_s64(&t.mm[a][slot], e);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// CTA-private group table in shared memory (BASELINE.json north_star: "group-by hashes into a shared-memory table reduced
// ... then a global atomic merge"; the reference keeps such key spaces in a dense array too:
// DictionaryBasedGroupKeyGenerator.java:285-414 ArrayBasedHolder, DoubleGroupByResultHolder.java:74-98).
// A dense table of S slots is replicated R times per CTA (warp w updates replica w % R): row counts are native 32-bit
// ATOMS, sums / min / max are 64-bit compare-and-swap loops on shared memory (SASS ATOMS.CAST.SPIN.64) -- an order of
// magnitude above the ~77 G/s of same-line L2 reductions that bounded the global-table kernel at 25 % selectivity.  At the
// end every CTA merges its non-empty slots into the global table with one RED per cell.
// Layout of one replica: cnt u32[S] | fcnt u32[n_fc][S] | acc u64[n_acc][S]   (acc: f64 sum, or order-encoded i64 min/max).
// ------------------------------------------------------------------------------------------------
// The cells are addressed in the shared STATE SPACE (32-bit addresses, atom.shared / red.shared / ld.shared PTX): through
// generic pointers the compiler emits generic ATOM.E instructions that resolve the address window at run time -- measured
// no faster than the L2 reductions they were meant to replace.
__device__ __forceinline__ void pb_sh_add_u32(uint32_t a, uint32_t v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t pb_sh_atom_add_u32(uint32_t a, uint32_t v) { uint32_t o; asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(o) : "r"(a), "r"(v) : "memory"); return o; }
__device__ __forceinline__ unsigned long long pb_sh_ld_u64(uint32_t a) { unsigned long long v; asm volatile("ld.volatile.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ uint32_t pb_sh_ld_u32(uint32_t a) { uint32_t v; asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void pb_sh_st_u64(uint32_t a, unsigned long long v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void pb_sh_st_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned long long pb_sh_cas_u64(uint32_t a, unsigned long long cmp, unsigned long long val) {
  unsigned long long old;
  asm volatile("atom.shared.cas.b64 %0, [%1], %2, %3;" : "=l"(old) : "r"(a), "l"(cmp), "l"(val) : "memory");
  return old;
}
struct SmemTable {
  uint32_t base;            // shared-space address of this warp's replica
  uint32_t S, n_fc;
  int8_t acc_of[PB_MAX_AGGS];   // aggregation -> accumulator array (SUM / AVG / MIN / MAX), -1 = none
  int8_t fc_of[PB_MAX_AGGS];    // aggregation -> filtered row counter (COUNT / AVG under a FILTER clause), -1 = none
  __device__ __forceinline__ uint32_t cnt(uint32_t slot) const { return base + 4u * slot; }
  __device__ __forceinline__ uint32_t fcnt(int k, uint32_t slot) const { return base + 4u * ((uint32_t)(1 + k) * S + slot); }
  __device__ __forceinline__ uint32_t acc(int k, uint32_t slot) const { return base + ((((1u + n_fc) * S * 4u) + 7u) & ~7u) + 8u * ((uint32_t)k * S + slot); }
};
__host__ __device__ __forceinline__ size_t pb_smem_table_bytes(uint32_t S, int n_fc, int n_acc) {
  return ((((size_t)(1 + n_fc) * S * 4 + 7) & ~(size_t)7) + (size_t)n_acc * S * 8 + 15) & ~(size_t)15;
}

__device__ __forceinline__ void pb_accumulate_smem(const DevQuery& Q, const DevSegQuery& sq, const DevTable& t, const SmemTable& st, uint32_t doc, uint32_t fpass) {
  const int nA = Q.n_aggs;
  uint64_t slot, slot_hi;
  double vals[PB_MAX_AGGS];
  pb_gather_doc(Q, sq, doc, slot, slot_hi, vals);
  const uint32_t sl = (uint32_t)slot;
  pb_sh_add_u32(st.cnt(sl), 1u);
  for (int a = 0; a < nA; a++) {
    const int op = Q.agg_op[a];
    const int fo = Q.agg_filter_of[a];
    if (fo >= 0) {
      if (!((fpass >> fo) & 1u)) continue;
      if (st.fc_of[a] >= 0) pb_sh_add_u32(st.fcnt(st.fc_of[a], sl), 1u);
    }
    if (op == 0) continue;
    const double v = vals[a];
    if (op == 5) {                               // distinct bitsets / value sets stay in global memory (idempotent: no contention cost)
      if (t.dset[a]) { pb_dset_insert(t, a, slot, (unsigned long long)__double_as_longlong(v)); continue; }
      uint32_t id = (uint32_t)__double_as_longlong(v);
      pb_red_or_b32(&t.dc_bits[a][slot * t.dc_words[a] + (id >> 5)], 1u << (id & 31));
      continue;
    }
    const uint32_t cell = st.acc(st.acc_of[a], sl);
    if (op == 1 || op == 4) {
      unsigned long long old = pb_sh_ld_u64(cell), assumed;
      do {
        assumed = old;
        old = pb_sh_cas_u64(cell, assumed, (unsigned long long)__double_as_longlong(__longlong_as_double((long long)assumed) + v));
      } while (old != assumed);
    } else if (v == v) {
      const long long e = op == 2 ? pb_enc_f64(v) : ~pb_enc_f64(v);
      long long old = (long long)pb_sh_ld_u64(cell);
      while (e < old) {                          // most docs do not improve the extreme: a plain load
        const long long seen = (long long)pb_sh_cas_u64(cell, (unsigned long long)old, (unsigned long long)e);
        if (seen == old) break;
        old = seen;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Kernel 1: pb_filter_kernel  (DocIdSetOperator + filter operators: SURVEY.md §3.2)
//
// A CTA owns a contiguous range of 1024-doc chunks; inside it every WARP is an independent worker with its
// own 2-stage TMA pipeline (cp.async.bulk + mbarrier) over its chunks — no block-wide barrier in the steady
// state.  Per unit: unpack + predicate tree on 32-bit doc masks (dense leaves), candidate leaves on the survivors, then the
// matching docIds go to the warp's output buffer (one ATOMG per ~256 matches reserves their place in the match list).
// ------------------------------------------------------------------------------------------------
struct __align__(16) FilterSmemHeader {
  uint64_t full[PB_NWARPS][PB_NSTAGE];
  uint32_t slot_stride[PB_MAX_SCAN_SLOTS];   // bytes of one work unit of the slot (U * 128 * bits)
  uint32_t slot_last_rel[PB_MAX_SCAN_SLOTS]; // first unit index whose load must be clipped to the buffer end
  uint32_t n_scan_full_bytes;                // expect_tx total of an unclipped unit
  int32_t flat_and;                          // program is AND(leaf, leaf, ...) (or a single leaf): no stack needed
  int32_t n_flat;
  int32_t flat_leaf[PB_MAX_LEAVES];
  int32_t n_dense;                           // flat_leaf[0 .. n_dense) run on the staged unit, the rest on the candidates
  int32_t pad_g;
  alignas(16) uint8_t seg[PB_SEG_FILTER_BYTES];   // the filter part of the current DevSegQuery
};

// U = 1024-doc chunks per work unit (one TMA load + one dispatch per predicate leaf per unit)
//
// SW / SPK: plan-time specialisation.  SW = 0 is the general kernel (any predicate tree, every width and predicate kind
// dispatched at run time: ~27 k SASS instructions, whose instruction-cache misses and dispatch cost were a fifth of the
// issue slots of the common case).  SW > 0 is a kernel for ONE shape -- a flat conjunction whose only streamed leaf is a
// dictionary column of SW bits tested with predicate kind SPK (0 = dictId range, 1 = IN / NOT IN membership LUT), every
// other leaf evaluated on the candidates -- with that leaf's unpack + test inlined and nothing else compiled in.  The host
// picks it when every segment of the launch has that shape (pb_filter_spec.cu holds the instantiations).
template <int U, int MIN_CTAS, int SW = 0, int SPK = 0>
__global__ void __launch_bounds__(PB_NTHREADS, MIN_CTAS) pb_filter_kernel(const __grid_constant__ DevQuery Q) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  FilterSmemHeader* H = reinterpret_cast<FilterSmemHeader*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint8_t* dyn = smem_raw + ((sizeof(FilterSmemHeader) + 127) & ~(size_t)127);
  uint8_t* set_cache = dyn;
  dyn += (Q.set_cache_bytes + 127) & ~127;
  uint16_t* cand = reinterpret_cast<uint16_t*>(dyn);     // per-warp candidate lists (only when some leaf is evaluated on candidates)
  dyn += Q.cand_bytes;
  const uint32_t OUT_CAP = (uint32_t)Q.out_cap, CAND_CAP = (uint32_t)Q.cand_cap;
  uint32_t* ob = reinterpret_cast<uint32_t*>(dyn) + (size_t)warp * OUT_CAP;   // this warp's output buffer
  dyn += (size_t)PB_NWARPS * OUT_CAP * sizeof(uint32_t);
  uint32_t out_n = 0;                                     // buffered matches (warp-uniform)
  auto flush_out = [&]() {
    if (out_n == 0) return;
    __syncwarp();
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(Q.match_count, (unsigned long long)out_n);
    base = __shfl_sync(0xffffffffu, base, 0);
    for (uint32_t i = (uint32_t)lane; i < out_n; i += 32) Q.match_list[base + i] = ob[i];
    __syncwarp();
    out_n = 0;
  };
  uint8_t* my_stages = dyn + (size_t)warp * PB_NSTAGE * Q.stage_bytes;
  const bool staged = Q.stage_bytes > 0;
  constexpr uint32_t UNIT_DOCS = U * PB_CHUNK_DOCS;

  if (lane == 0)
    for (int s = 0; s < PB_NSTAGE; s++) pb_mbar_init(&H->full[warp][s], 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  // this CTA's contiguous range of work units
  const uint64_t per = (Q.n_units + gridDim.x - 1) / gridDim.x;
  const uint64_t cta_lo = Q.unit_lo + (uint64_t)blockIdx.x * per;
  const uint64_t cta_hi = cta_lo + per < Q.unit_lo + Q.n_units ? cta_lo + per : Q.unit_lo + Q.n_units;
  if (cta_lo >= cta_hi) return;
  int seg_first = 0;
  while (seg_first + 1 < Q.n_segs && cta_lo >= Q.segs[seg_first + 1].unit_begin) seg_first++;

  uint32_t consumed = 0;   // units this warp has consumed so far: stage = consumed % NSTAGE, parity from consumed / NSTAGE
  const DevSegQuery& sq = *reinterpret_cast<const DevSegQuery*>(H->seg);   // only the filter part is valid
  const uint64_t l2_stream = pb_policy_evict_first();

  // evaluate one filter leaf on the staged unit: m[u] = this lane's 32-doc mask of sub-chunk u.  With sparse == true only
  // the docs still set in restrict_to[u] matter (AND chain with few survivors): decode just them.
  auto eval_leaf = [&](const DevLeaf& lf, const uint8_t* stage, uint64_t unit_doc0, int nu, const uint32_t* restrict_to, bool sparse, uint32_t* m) {
    switch (lf.kind) {
      case L_TRUE: for (int u = 0; u < nu; u++) m[u] = 0xffffffffu; return;
      case L_FALSE: for (int u = 0; u < nu; u++) m[u] = 0u; return;
      case L_DICT_RANGE: {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(stage + Q.slot_off[lf.slot]);
        PredRange pr; pr.lo = lf.lo; pr.span = lf.span;
        if (sparse) { for (int u = 0; u < nu; u++) m[u] = pb_eval_dict_sparse<PredRange>(p + u * 32 * lf.bits, lf.bits, pr, lane, restrict_to[u]); return; }
        pb_eval_dict<PredRange>(p, lf.bits, pr, lane, Q.generic, nu, m);
        return;
      }
      case L_DICT_SET: {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(stage + Q.slot_off[lf.slot]);
        if (lf.set_smem_off >= 0) {
          PredLut8 pl; pl.lut = set_cache + lf.set_smem_off;
          if (sparse) { for (int u = 0; u < nu; u++) m[u] = pb_eval_dict_sparse<PredLut8>(p + u * 32 * lf.bits, lf.bits, pl, lane, restrict_to[u]); return; }
          pb_eval_dict<PredLut8>(p, lf.bits, pl, lane, Q.generic, nu, m);
          return;
        }
        PredBits pb; pb.bits = lf.set_bits; pb.excl = (uint32_t)lf.exclusive;
        if (sparse) { for (int u = 0; u < nu; u++) m[u] = pb_eval_dict_sparse<PredBits>(p + u * 32 * lf.bits, lf.bits, pb, lane, restrict_to[u]); return; }
        pb_eval_dict<PredBits>(p, lf.bits, pb, lane, Q.generic, nu, m);
        return;
      }
      case L_RAW_RANGE_I:
      case L_RAW_RANGE_F:
      case L_RAW_SET: {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(stage + Q.slot_off[lf.slot]);
        for (int u = 0; u < nu; u++) m[u] = pb_eval_raw(p + u * (PB_CHUNK_DOCS / 4) * lf.raw_width, lf, lane);
        return;
      }
      default: {   // L_BITMAP (padded to whole units)
        for (int u = 0; u < nu; u++) {
          uint32_t w = __ldg(lf.bitmap + (unit_doc0 >> 5) + u * 32 + lane);
          m[u] = lf.exclusive ? ~w : w;
        }
        return;
      }
    }
  };

  for (int sgi = seg_first; sgi < Q.n_segs; sgi++) {
    if (Q.segs[sgi].unit_begin >= cta_hi) break;
    // ---- segment entry: filter descriptor, derived constants and LUTs into shared memory ----
    __syncthreads();   // everyone has left the previous segment
    {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(&Q.segs[sgi]);
      uint32_t* dst = reinterpret_cast<uint32_t*>(H->seg);
      for (int i = tid; i < (int)(PB_SEG_FILTER_BYTES / 4); i += PB_NTHREADS) dst[i] = src[i];
      __syncthreads();
      if (tid < sq.n_scan) {
        const uint32_t stride = (uint32_t)(UNIT_DOCS / 8) * (uint32_t)sq.scan[tid].bits_per_doc;
        H->slot_stride[tid] = stride;
        // units rel < last_rel can load stride + 16 bytes without leaving the (16-byte padded) buffer
        const uint64_t total = sq.scan[tid].bytes_total;
        H->slot_last_rel[tid] = total >= (uint64_t)stride + 16 ? (uint32_t)((total - stride - 16) / stride) + 1 : 0u;
      }
      if (tid == 96) {
        uint32_t t = 0;
        for (int c = 0; c < sq.n_scan; c++) t += (uint32_t)(UNIT_DOCS / 8) * (uint32_t)sq.scan[c].bits_per_doc + 16;
        H->n_scan_full_bytes = t;
      }
      if (tid == 64) {
        // flat conjunction?  postfix == leaf* AND(n)   or a single leaf   or empty (match all)
        int nl = 0; bool flat = true;
        for (int n = 0; n < sq.n_nodes; n++) {
          if (sq.node_kind[n] == N_LEAF) { if (nl < PB_MAX_LEAVES) H->flat_leaf[nl] = sq.node_arg[n]; nl++; }
          else if (!(sq.node_kind[n] == N_AND && n == sq.n_nodes - 1 && sq.node_arg[n] == nl)) flat = false;
        }
        // most selective leaf first (insertion sort on the host's estimate); leaves evaluated on candidates go last
        int nd = 0;
        if (flat && nl <= PB_MAX_LEAVES) {
          auto key = [&](int l) { return sq.leaves[l].est_permille + (sq.leaves[l].gather ? 4096 : 0); };
          for (int a = 1; a < nl; a++) {
            int x = H->flat_leaf[a]; int b = a - 1;
            while (b >= 0 && key(H->flat_leaf[b]) > key(x)) { H->flat_leaf[b + 1] = H->flat_leaf[b]; b--; }
            H->flat_leaf[b + 1] = x;
          }
          for (int a = 0; a < nl; a++) if (!sq.leaves[H->flat_leaf[a]].gather) nd++;
        }
        H->flat_and = flat ? 1 : 0;
        H->n_flat = nl;
        H->n_dense = nd;
      }
      for (int l = 0; l < PB_MAX_LEAVES; l++) {
        const DevLeaf& lf = sq.leaves[l];
        if (lf.kind == L_DICT_SET && lf.set_smem_off >= 0) {
          // membership bytes with the exclusive flag (NOT_IN / NEQ) folded in
          for (int i = tid; i < lf.set_card; i += PB_NTHREADS)
            set_cache[lf.set_smem_off + i] = (uint8_t)(((__ldg(lf.set_bits + (i >> 5)) >> (i & 31)) & 1u) ^ (uint32_t)lf.exclusive);
        }
      }
      __syncthreads();
    }
    const uint64_t seg_lo = sq.unit_begin > cta_lo ? sq.unit_begin : cta_lo;
    const uint64_t seg_end = sq.unit_begin + sq.n_units;
    const uint64_t seg_hi = seg_end < cta_hi ? seg_end : cta_hi;
    // this warp's units in this segment: seg_lo + warp, + NWARPS, ...
    const uint64_t first = seg_lo + warp;
    const uint32_t n_mine = first < seg_hi ? (uint32_t)((seg_hi - first + PB_NWARPS - 1) / PB_NWARPS) : 0u;
    const uint32_t rel0 = (uint32_t)(first - sq.unit_begin);     // unit index inside the segment
    const int n_scan = sq.n_scan;
    unsigned long long matched = 0;
    uint32_t min_last_rel = 0xffffffffu;               // first unit whose load must be clipped to the buffer end
    for (int c = 0; c < n_scan; c++) min_last_rel = min(min_last_rel, H->slot_last_rel[c]);

    // producer side (lane 0 of each warp): load this warp's k-th unit of the segment into its stage
    auto issue = [&](uint32_t k, uint32_t seq) {
      const uint32_t rel = rel0 + k * PB_NWARPS;
      const int st = (int)(seq % PB_NSTAGE);
      uint8_t* dst = my_stages + (size_t)st * Q.stage_bytes;
      uint64_t* bar = &H->full[warp][st];
      if (__builtin_expect(rel < min_last_rel, 1)) {    // steady state: constant sizes
        pb_mbar_expect_tx(bar, H->n_scan_full_bytes);
        for (int c = 0; c < n_scan; c++) {
          const uint32_t stride = H->slot_stride[c];
          pb_tma_load_1d_hint(dst + Q.slot_off[c], sq.scan[c].base + (uint64_t)rel * stride, stride + 16, bar, l2_stream);
        }
        return;
      }
      uint32_t total = 0;
      uint32_t nbytes[PB_MAX_SCAN_SLOTS];
      for (int c = 0; c < n_scan; c++) {
        const uint64_t off = (uint64_t)rel * H->slot_stride[c];                   // unit starts are 128-byte multiples
        const uint64_t want = (uint64_t)H->slot_stride[c] + 16;                   // +16: the word after the unit
        const uint64_t avail = sq.scan[c].bytes_total - off;
        nbytes[c] = (uint32_t)((want < avail ? want : avail) & ~(uint64_t)15);
        total += nbytes[c];
      }
      pb_mbar_expect_tx(bar, total);
      for (int c = 0; c < n_scan; c++)
        pb_tma_load_1d(dst + Q.slot_off[c], sq.scan[c].base + (uint64_t)rel * H->slot_stride[c], nbytes[c], bar);
    };

    if (staged && Q.use_tma && lane == 0)
      for (uint32_t k = 0; k < PB_NSTAGE - 1 && k < n_mine; k++) issue(k, consumed + k);

    for (uint32_t k = 0; k < n_mine; k++) {
      const uint64_t unit_doc0 = (uint64_t)(rel0 + k * PB_NWARPS) * UNIT_DOCS;
      const int st = (int)(consumed % PB_NSTAGE);
      uint8_t* stage = my_stages + (size_t)st * Q.stage_bytes;
      if (staged) {
        if (__builtin_expect(Q.use_tma != 0, 1)) {
          // the stage being refilled was consumed one iteration ago by this same warp
          if (lane == 0 && k + PB_NSTAGE - 1 < n_mine) issue(k + PB_NSTAGE - 1, consumed + PB_NSTAGE - 1);
          pb_mbar_wait(&H->full[warp][st], (consumed / PB_NSTAGE) & 1u);
        } else {
          for (int c = 0; c < n_scan; c++) {
            const uint64_t off = (uint64_t)(rel0 + k * PB_NWARPS) * H->slot_stride[c];
            const uint64_t want = (uint64_t)H->slot_stride[c] + 16;
            const uint64_t avail = sq.scan[c].bytes_total - off;
            const uint64_t n = (want < avail ? want : avail) & ~(uint64_t)15;
            const uint4* s4 = reinterpret_cast<const uint4*>(sq.scan[c].base + off);
            uint4* d4 = reinterpret_cast<uint4*>(stage + Q.slot_off[c]);
            for (uint32_t i = lane; i < (uint32_t)(n / 16); i += 32) d4[i] = __ldg(s4 + i);
          }
          __syncwarp();
        }
      }
      consumed++;

      // ---- predicate tree on 32-doc masks (one mask word per lane per sub-chunk) ----
      uint32_t mask[U], tmp[U];
      int nu = 0;
      const uint32_t nd_rel = (uint32_t)sq.num_docs - (uint32_t)unit_doc0;      // docs from the start of this unit (>= 1; docs of a segment fit 31 bits)
      nu = nd_rel >= (uint32_t)U * PB_CHUNK_DOCS ? U : (int)((nd_rel + PB_CHUNK_DOCS - 1) / PB_CHUNK_DOCS);
#pragma unroll
      for (int u = 0; u < U; u++) {
        const uint32_t d = (uint32_t)u * PB_CHUNK_DOCS + 32u * (uint32_t)lane;
        mask[u] = nd_rel >= d + 32u ? 0xffffffffu : (nd_rel <= d ? 0u : ((1u << (nd_rel - d)) - 1u));
      }
      const int n_cand_leaves = H->flat_and ? H->n_flat - H->n_dense : 0;
      if constexpr (SW > 0) {
        // the one streamed leaf, unpack + predicate inlined for this width and kind
        const DevLeaf& lf = sq.leaves[H->flat_leaf[0]];
        const uint32_t* p = reinterpret_cast<const uint32_t*>(stage + Q.slot_off[lf.slot]);
        if constexpr (SPK == 0) {
          PredRange pr; pr.lo = lf.lo; pr.span = lf.span;
#pragma unroll
          for (int u = 0; u < U; u++) if (u < nu) mask[u] &= pb_eval_dict_w<SW, PredRange>(p + u * 32 * SW, pr, lane);
        } else {
          PredLut8 pl; pl.lut = set_cache + lf.set_smem_off;
#pragma unroll
          for (int u = 0; u < U; u++) if (u < nu) mask[u] &= pb_eval_dict_w<SW, PredLut8>(p + u * 32 * SW, pl, lane);
        }
      } else if (__builtin_expect(H->flat_and != 0, 1)) {
        const int nl = H->n_dense;
        for (int i = 0; i < nl; i++) {
          // few survivors in the whole unit -> restricted scan of the remaining leaves (leaves arrive ordered by
          // estimated selectivity from the host)
          uint32_t pc = 0;
#pragma unroll
          for (int u = 0; u < U; u++) pc += (uint32_t)__popc(mask[u]);
          const bool sparse = i > 0 && !Q.generic && __reduce_add_sync(0xffffffffu, pc) <= (uint32_t)Q.sparse_max * U;
          eval_leaf(sq.leaves[H->flat_leaf[i]], stage, unit_doc0, nu, mask, sparse, tmp);
          uint32_t any = 0;
#pragma unroll
          for (int u = 0; u < U; u++) { if (u < nu) mask[u] &= tmp[u]; any |= mask[u]; }
          if (sparse && !__any_sync(0xffffffffu, any != 0)) break;
        }
      } else {
        uint32_t stack[PB_MAX_LEAVES][U];
        const uint32_t all[2] = {0xffffffffu, 0xffffffffu};
        int sp = 0;
        for (int n = 0; n < sq.n_nodes; n++) {
          const int kind = sq.node_kind[n], arg = sq.node_arg[n];
          if (kind == N_LEAF) { eval_leaf(sq.leaves[arg], stage, unit_doc0, nu, all, false, stack[sp]); sp++; }
          else if (kind == N_NOT) { for (int u = 0; u < nu; u++) stack[sp - 1][u] = ~stack[sp - 1][u]; }
          else {
            for (int u = 0; u < nu; u++) {
              uint32_t r = stack[sp - arg][u];
              for (int i = 1; i < arg; i++) r = (kind == N_AND) ? (r & stack[sp - arg + i][u]) : (r | stack[sp - arg + i][u]);
              stack[sp - arg][u] = r;
            }
            sp -= arg - 1;
          }
        }
        if (sp > 0) for (int u = 0; u < nu; u++) mask[u] &= stack[0][u];
      }
      __syncwarp();   // all lanes are done reading this stage before lane 0 may refill it next iteration

      // ---- append the matching docIds (global doc numbering) to the match list ----
      // Matches go through a per-warp output buffer in shared memory and reach the global list in batches: one
      // ATOMG (whose ~1 us round trip used to sit on every unit's critical path) per ~PB_OUT_CAP matches.
      uint32_t cnt = 0;
#pragma unroll
      for (int u = 0; u < U; u++) cnt += (uint32_t)__popc(mask[u]);
      const uint32_t mx = __reduce_max_sync(0xffffffffu, cnt);
      if (mx == 0) continue;                                   // warp-uniform
      uint32_t excl = 0, total = 0;
      const uint32_t lt = (1u << lane) - 1u;
      if (mx <= 4) {
        // few matches per lane: exclusive prefix from ballots (no shuffle dependency chain)
        for (uint32_t kk = 1; kk <= mx; kk++) {
          const uint32_t b = __ballot_sync(0xffffffffu, cnt >= kk);
          excl += __popc(b & lt);
          total += __popc(b);
        }
      } else {
        uint32_t incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        total = __shfl_sync(0xffffffffu, incl, 31);
        excl = incl - cnt;
      }
      const uint32_t gunit0 = (uint32_t)(sq.doc_base + unit_doc0);
      if (n_cand_leaves == 0) {
        if (__builtin_expect(total > OUT_CAP, 0)) {
          // dense matches: straight to the list
          unsigned long long base = 0;
          if (lane == 0) base = atomicAdd(Q.match_count, (unsigned long long)total);
          base = __shfl_sync(0xffffffffu, base, 0);
          uint32_t* out = Q.match_list + base + excl;
#pragma unroll
          for (int u = 0; u < U; u++) {
            const uint32_t gdoc0 = gunit0 + (uint32_t)u * PB_CHUNK_DOCS + 32u * (uint32_t)lane;
            uint32_t mm = mask[u];
            while (mm) {
              const int bit = __ffs(mm) - 1;
              mm &= mm - 1;
              *out++ = gdoc0 + (uint32_t)bit;
            }
          }
        } else {
          if (out_n + total > OUT_CAP) flush_out();
          uint32_t* out = ob + out_n + excl;
#pragma unroll
          for (int u = 0; u < U; u++) {
            const uint32_t gdoc0 = gunit0 + (uint32_t)u * PB_CHUNK_DOCS + 32u * (uint32_t)lane;
            uint32_t mm = mask[u];
            while (mm) {
              const int bit = __ffs(mm) - 1;
              mm &= mm - 1;
              *out++ = gdoc0 + (uint32_t)bit;
            }
          }
          out_n += total;
        }
        matched += total;
      } else {
        // ---- candidates: survivors of the staged leaves, compacted into this warp's list, then one lane per candidate
        // tests the remaining leaves straight from their forward indexes (all 32 gathers of a round in flight at once) ----
        uint16_t* cl = cand + (size_t)warp * CAND_CAP;
        for (uint32_t pass0 = 0; pass0 < total; pass0 += CAND_CAP) {     // one pass unless the estimate was far off
          if (pass0) __syncwarp();
          {
            uint32_t pos = excl - pass0;                                     // (wraps below the window: unsigned compare)
#pragma unroll
            for (int u = 0; u < U; u++) {
              const uint32_t off0 = (uint32_t)u * PB_CHUNK_DOCS + 32u * (uint32_t)lane;
              uint32_t mm = mask[u];
              while (mm) {
                const int bit = __ffs(mm) - 1;
                mm &= mm - 1;
                if (pos < CAND_CAP) cl[pos] = (uint16_t)(off0 + (uint32_t)bit);
                pos++;
              }
            }
          }
          __syncwarp();
          const uint32_t n_pass = total - pass0 < CAND_CAP ? total - pass0 : CAND_CAP;
          for (uint32_t b0 = 0; b0 < n_pass; b0 += 32) {
            const uint32_t idx = b0 + (uint32_t)lane;
            bool alive = idx < n_pass;
            const uint32_t off = alive ? (uint32_t)cl[idx] : 0u;
            const uint32_t doc = (uint32_t)unit_doc0 + off;          // doc inside the segment
            for (int i = 0; i < n_cand_leaves; i++) {
              if (alive) alive = pb_leaf_test_doc(sq.leaves[H->flat_leaf[H->n_dense + i]], set_cache, doc);
              if (!__any_sync(0xffffffffu, alive)) break;
            }
            const uint32_t bal = __ballot_sync(0xffffffffu, alive);
            if (bal) {
              const uint32_t n = (uint32_t)__popc(bal);
              if (out_n + n > OUT_CAP) flush_out();
              if (alive) ob[out_n + __popc(bal & lt)] = gunit0 + off;
              out_n += n;
              matched += n;
            }
          }
        }
        __syncwarp();   // the list is rewritten by the next unit
      }
    }
    flush_out();
    // ---- segment exit: numDocsScanned of this segment's table (matched is warp-uniform) ----
    if (lane == 0 && matched && !Q.agg_counts_docs) pb_red_add_u64(Q.tables[sq.table].docs_matched, matched);
  }
}

// ------------------------------------------------------------------------------------------------
// Kernel 2: pb_agg_kernel  (ProjectionOperator + GroupByOperator / AggregationOperator: SURVEY.md §3.1)
//
// One thread per matching doc, grid-strided over the match list written by pb_filter_kernel (or over all docs
// when there is no filter).  Each thread gathers the group-key / metric dictIds of its doc straight from the
// bit-packed forward indexes in HBM (only the sectors holding matching rows are touched), decodes through the
// dictionary, and reduces into the table with native L2 reductions.  With every match in flight at once the
// dependent-load latency of the gathers is hidden by thread-level parallelism.
// ------------------------------------------------------------------------------------------------
#define PB_AGG_MAX_SEGS_SMEM 1024

template <int MIN_CTAS>
__global__ void __launch_bounds__(PB_NTHREADS, MIN_CTAS) pb_agg_kernel(const __grid_constant__ DevQuery Q) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __shared__ unsigned long long s_doc_base[PB_AGG_MAX_SEGS_SMEM + 1];
  __shared__ unsigned long long s_red_u64[PB_NWARPS];
  __shared__ double s_red_f64[PB_NWARPS];
  __shared__ long long s_red_i64[PB_NWARPS];
  __shared__ int s_table0;
  const int n_segs = Q.n_segs;
  const int n_smem = n_segs < PB_AGG_MAX_SEGS_SMEM ? n_segs : PB_AGG_MAX_SEGS_SMEM;
  for (int i = tid; i < n_smem; i += PB_NTHREADS) s_doc_base[i] = Q.segs[i].doc_base;
  KeylessAcc ka;
  ka.sum = nullptr; ka.mm = nullptr; ka.cnt = nullptr;
  const long long ENC_POS_INF = 0x7ff0000000000000LL;
  const long long ENC_NEG_INF = (long long)0xfff0000000000000ULL ^ 0x7fffffffffffffffLL;
  const bool keyless = Q.table_mode == T_KEYLESS;
  if (keyless) {
    ka.sum = reinterpret_cast<double*>(smem_raw);
    ka.mm = reinterpret_cast<long long*>(smem_raw + sizeof(double) * Q.n_aggs * PB_NTHREADS);
    if (Q.n_agg_filters > 0) ka.cnt = reinterpret_cast<unsigned long long*>(smem_raw + 2 * sizeof(double) * Q.n_aggs * PB_NTHREADS);
    for (int a = 0; a < Q.n_aggs; a++) {
      ka.sum[a * PB_NTHREADS + tid] = 0.0;
      ka.mm[a * PB_NTHREADS + tid] = Q.agg_op[a] == 2 ? ENC_POS_INF : ENC_NEG_INF;
      if (ka.cnt) ka.cnt[a * PB_NTHREADS + tid] = 0ull;
    }
  }
  __syncthreads();

  if (Q.phase == 2 && *Q.any_limit == 0) return;          // repair pass: nothing was refused, nothing to repair
  const unsigned long long n = Q.match_all ? Q.n_docs_total : *Q.match_count;
  unsigned long long keyless_rows = 0;
  int my_table = -1;      // keyless: table the private accumulators currently belong to

  auto keyless_flush_thread = [&]() {   // rare path: this thread moves on to another table
    if (my_table < 0) return;
    const DevTable& t = Q.tables[my_table];
    if (keyless_rows) pb_red_add_u64(&t.rowcnt[0], keyless_rows);
    keyless_rows = 0;
    for (int a = 0; a < Q.n_aggs; a++) {
      const int op = Q.agg_op[a];
      if (op == 1 || op == 4) { pb_red_add_f64(&t.sum[a][0], ka.sum[a * PB_NTHREADS + tid]); ka.sum[a * PB_NTHREADS + tid] = 0.0; }
      else if (op == 2) { pb_red_min_s64(&t.mm[a][0], ka.mm[a * PB_NTHREADS + tid]); ka.mm[a * PB_NTHREADS + tid] = ENC_POS_INF; }
      else if (op == 3) { pb_red_min_s64(&t.mm[a][0], ~ka.mm[a * PB_NTHREADS + tid]); ka.mm[a * PB_NTHREADS + tid] = ENC_NEG_INF; }
      if (ka.cnt && t.fcnt[a]) { if (ka.cnt[a * PB_NTHREADS + tid]) pb_red_add_u64(&t.fcnt[a][0], ka.cnt[a * PB_NTHREADS + tid]); ka.cnt[a * PB_NTHREADS + tid] = 0ull; }
    }
  };
  // swim-lane statistics: docs of the current segment that reached this kernel [0] / passed clause f [1 + f], kept per
  // thread and flushed when the thread moves to another segment
  const int nF = Q.n_agg_filters;
  int stat_seg = -1;
  unsigned int stat_cnt[1 + PB_MAX_AGG_FILTERS];
#pragma unroll
  for (int f = 0; f <= PB_MAX_AGG_FILTERS; f++) stat_cnt[f] = 0;
  auto stat_flush = [&]() {
    if (stat_seg < 0) return;
    unsigned long long* dst = Q.segs[stat_seg].af_docs;
#pragma unroll
    for (int f = 0; f <= PB_MAX_AGG_FILTERS; f++) if (f <= nF && stat_cnt[f]) { pb_red_add_u64(dst + f, (unsigned long long)stat_cnt[f]); stat_cnt[f] = 0; }
  };

  for (unsigned long long i = (unsigned long long)blockIdx.x * PB_NTHREADS + tid; i < n; i += (unsigned long long)gridDim.x * PB_NTHREADS) {
    const unsigned long long gdoc = Q.match_all ? i : (unsigned long long)__ldg(Q.match_list + i);
    // segment of this doc: last doc_base <= gdoc
    int lo = 0, hi = n_segs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      const unsigned long long b = mid < PB_AGG_MAX_SEGS_SMEM ? s_doc_base[mid] : Q.segs[mid].doc_base;
      if (b <= gdoc) lo = mid; else hi = mid - 1;
    }
    const DevSegQuery& sg = Q.segs[lo];
    const uint32_t doc = (uint32_t)(gdoc - (lo < PB_AGG_MAX_SEGS_SMEM ? s_doc_base[lo] : sg.doc_base));
    const int table = sg.table;
    if (keyless && table != my_table) { keyless_flush_thread(); my_table = table; }
    uint32_t fpass = 0;
    if (nF > 0) {
      fpass = pb_agg_filter_bits(sg, doc);
      if (lo != stat_seg) { stat_flush(); stat_seg = lo; }
      stat_cnt[0]++;
#pragma unroll
      for (int f = 0; f < PB_MAX_AGG_FILTERS; f++) if (f < nF) stat_cnt[1 + f] += (fpass >> f) & 1u;
    }
    pb_accumulate(Q, sg, Q.tables[table], doc, ka, keyless_rows, fpass);
  }
  if (nF > 0) stat_flush();

  if (!keyless) return;
  // ---- keyless: merge the private accumulators; one reduction per CTA when the whole CTA saw one table ----
  if (tid == 0) s_table0 = -1;
  __syncthreads();
  if (my_table >= 0) atomicMax(&s_table0, my_table);
  __syncthreads();
  const int t0 = s_table0;
  const int uniform = __syncthreads_and(my_table < 0 || my_table == t0);
  if (!uniform || t0 < 0) { keyless_flush_thread(); return; }
  const DevTable& t = Q.tables[t0];
  unsigned long long r = keyless_rows;
  for (int o = 16; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
  if (lane == 0) s_red_u64[warp] = r;
  __syncthreads();
  if (tid == 0) { unsigned long long tot = 0; for (int w = 0; w < PB_NWARPS; w++) tot += s_red_u64[w]; if (tot) pb_red_add_u64(&t.rowcnt[0], tot); }
  for (int a = 0; a < Q.n_aggs; a++) {
    const int op = Q.agg_op[a];
    if (ka.cnt && t.fcnt[a]) {
      unsigned long long c = ka.cnt[a * PB_NTHREADS + tid];
      for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
      if (lane == 0) s_red_u64[warp] = c;
      __syncthreads();
      if (tid == 0) { unsigned long long tot = 0; for (int w = 0; w < PB_NWARPS; w++) tot += s_red_u64[w]; if (tot) pb_red_add_u64(&t.fcnt[a][0], tot); }
      __syncthreads();
    }
    if (op == 1 || op == 4) {
      double v = ka.sum[a * PB_NTHREADS + tid];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
      if (lane == 0) s_red_f64[warp] = v;
      __syncthreads();
      if (tid == 0) { double tot = 0; for (int w = 0; w < PB_NWARPS; w++) tot += s_red_f64[w]; pb_red_add_f64(&t.sum[a][0], tot); }
      __syncthreads();
    } else if (op == 2 || op == 3) {
      long long v = ka.mm[a * PB_NTHREADS + tid];
      for (int o = 16; o > 0; o >>= 1) { long long u = __shfl_down_sync(0xffffffffu, v, o); v = (op == 2) ? (u < v ? u : v) : (u > v ? u : v); }
      if (lane == 0) s_red_i64[warp] = v;
      __syncthreads();
      if (tid == 0) {
        long long tot = s_red_i64[0];
        for (int w = 1; w < PB_NWARPS; w++) { long long u = s_red_i64[w]; tot = (op == 2) ? (u < tot ? u : tot) : (u > tot ? u : tot); }
        pb_red_min_s64(&t.mm[a][0], op == 2 ? tot : ~tot);
      }
      __syncthreads();
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Kernel 2b: pb_agg_smem_kernel — pb_agg_kernel for ONE dense table whose slots fit shared memory: one CTA of 1024 threads
// per SM, CTA-private replicas of the table (see SmemTable), one merge into the global table at the end.  With few matches
// (< st_min_docs, known on the device only) it updates the global table directly like pb_agg_kernel.
// ------------------------------------------------------------------------------------------------
#define PB_AGG_SMEM_THREADS 1024
static __global__ void __launch_bounds__(PB_AGG_SMEM_THREADS, 1) pb_agg_smem_kernel(const __grid_constant__ DevQuery Q) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ unsigned long long s_doc_base[PB_AGG_MAX_SEGS_SMEM + 1];
  const int tid = threadIdx.x, warp = tid >> 5;
  const int n_segs = Q.n_segs;
  const int n_smem = n_segs < PB_AGG_MAX_SEGS_SMEM ? n_segs : PB_AGG_MAX_SEGS_SMEM;
  for (int i = tid; i < n_smem; i += PB_AGG_SMEM_THREADS) s_doc_base[i] = Q.segs[i].doc_base;
  const unsigned long long n = Q.match_all ? Q.n_docs_total : *Q.match_count;
  const DevTable& t = Q.tables[0];
  const uint32_t S = (uint32_t)Q.st_slots, R = (uint32_t)Q.st_replicas;
  SmemTable st;
  st.S = S;
  int n_acc = 0, n_fc = 0;
  for (int a = 0; a < PB_MAX_AGGS; a++) {
    const int op = a < Q.n_aggs ? Q.agg_op[a] : 0;
    st.acc_of[a] = (a < Q.n_aggs && op >= 1 && op <= 4) ? (int8_t)n_acc++ : (int8_t)-1;
    st.fc_of[a] = (a < Q.n_aggs && Q.agg_filter_of[a] >= 0 && t.fcnt[a] != nullptr) ? (int8_t)n_fc++ : (int8_t)-1;
  }
  st.n_fc = (uint32_t)n_fc;
  const size_t rep_bytes = pb_smem_table_bytes(S, n_fc, n_acc);
  const uint32_t smem0 = pb_smem_u32(smem_raw);
  st.base = smem0 + ((uint32_t)warp & (R - 1)) * (uint32_t)rep_bytes;
  const bool use_smem = n >= Q.st_min_docs;
  if (use_smem) {
    for (uint32_t r = 0; r < R; r++) {
      SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes;
      for (uint32_t i = tid; i < (1 + (uint32_t)n_fc) * S; i += PB_AGG_SMEM_THREADS) pb_sh_st_u32(z.cnt(i), 0u);
      for (int a = 0; a < Q.n_aggs; a++) {
        if (st.acc_of[a] < 0) continue;
        const unsigned long long init = (Q.agg_op[a] == 1 || Q.agg_op[a] == 4) ? 0ull : 0x7fffffffffffffffull;
        for (uint32_t i = tid; i < S; i += PB_AGG_SMEM_THREADS) pb_sh_st_u64(z.acc(st.acc_of[a], i), init);
      }
    }
  }
  __syncthreads();

  const int nF = Q.n_agg_filters;
  int stat_seg = -1;
  unsigned int stat_cnt[1 + PB_MAX_AGG_FILTERS];
#pragma unroll
  for (int f = 0; f <= PB_MAX_AGG_FILTERS; f++) stat_cnt[f] = 0;
  auto stat_flush = [&]() {
    if (stat_seg < 0) return;
    unsigned long long* dst = Q.segs[stat_seg].af_docs;
#pragma unroll
    for (int f = 0; f <= PB_MAX_AGG_FILTERS; f++) if (f <= nF && stat_cnt[f]) { pb_red_add_u64(dst + f, (unsigned long long)stat_cnt[f]); stat_cnt[f] = 0; }
  };
  KeylessAcc ka; ka.sum = nullptr; ka.mm = nullptr; ka.cnt = nullptr;
  unsigned long long unused_rows = 0;

  for (unsigned long long i = (unsigned long long)blockIdx.x * PB_AGG_SMEM_THREADS + tid; i < n; i += (unsigned long long)gridDim.x * PB_AGG_SMEM_THREADS) {
    const unsigned long long gdoc = Q.match_all ? i : (unsigned long long)__ldg(Q.match_list + i);
    int lo = 0, hi = n_segs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      const unsigned long long b = mid < PB_AGG_MAX_SEGS_SMEM ? s_doc_base[mid] : Q.segs[mid].doc_base;
      if (b <= gdoc) lo = mid; else hi = mid - 1;
    }
    const DevSegQuery& sg = Q.segs[lo];
    const uint32_t doc = (uint32_t)(gdoc - (lo < PB_AGG_MAX_SEGS_SMEM ? s_doc_base[lo] : sg.doc_base));
    uint32_t fpass = 0;
    if (nF > 0) {
      fpass = pb_agg_filter_bits(sg, doc);
      if (lo != stat_seg) { stat_flush(); stat_seg = lo; }
      stat_cnt[0]++;
#pragma unroll
      for (int f = 0; f < PB_MAX_AGG_FILTERS; f++) if (f < nF) stat_cnt[1 + f] += (fpass >> f) & 1u;
    }
    if (use_smem) pb_accumulate_smem(Q, sg, t, st, doc, fpass);
    else pb_accumulate(Q, sg, t, doc, ka, unused_rows, fpass);
  }
  if (nF > 0) stat_flush();
  if (!use_smem) return;
  __syncthreads();
  // ---- merge the CTA's replicas into the global table: one RED per non-empty cell ----
  for (uint32_t i = tid; i < S; i += PB_AGG_SMEM_THREADS) {
    unsigned long long c = 0;
    for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; c += pb_sh_ld_u32(z.cnt(i)); }
    if (c == 0) continue;
    pb_red_add_u64(&t.rowcnt[i], c);
    for (int a = 0; a < Q.n_aggs; a++) {
      if (st.fc_of[a] >= 0) {
        unsigned long long fc = 0;
        for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; fc += pb_sh_ld_u32(z.fcnt(st.fc_of[a], i)); }
        if (fc) pb_red_add_u64(&t.fcnt[a][i], fc);
      }
      if (st.acc_of[a] < 0) continue;
      const int op = Q.agg_op[a];
      if (op == 1 || op == 4) {
        double v = 0.0;
        for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; v += __longlong_as_double((long long)pb_sh_ld_u64(z.acc(st.acc_of[a], i))); }
        pb_red_add_f64(&t.sum[a][i], v);
      } else {
        long long m = 0x7fffffffffffffffLL;
        for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; const long long o = (long long)pb_sh_ld_u64(z.acc(st.acc_of[a], i)); m = o < m ? o : m; }
        if (m != 0x7fffffffffffffffLL) pb_red_min_s64(&t.mm[a][i], m);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Kernel 2c: pb_agg_rows_kernel — the aggregation of the common query shape, specialised at plan time: a dense group table
// whose keys are dictionary columns and whose aggregation inputs are COUNT(*) or numeric columns, every one of them a field
// of the segments' ROW GROUPS (dictIds for the keys, decoded values for the inputs).  A matching doc is then one row: no
// per-column descriptors, no dictionary lookups, no bounds checks -- ~90 instructions per doc instead of the ~400 of the
// general kernel, which was instruction- and latency-bound (ncu, profiles/r2_kernels.md).  RW = 32-bit words per row.
// Table update: the CTA-private shared-memory table (SmemTable) when the launch carries one and has enough matches, else
// reductions into the global table.  Residual filter leaves (DevRowLeaf) are tested on the row before either.
// ------------------------------------------------------------------------------------------------
struct DevRowKey { uint32_t off, bits; uint64_t mult; const int32_t* remap; };
struct DevRowAgg { uint32_t off, width, type, exact_int; };  // width 4 / 8 bytes, type PB_INT .. PB_DOUBLE; unused for COUNT(*).  exact_int: SUM / AVG
                                                             // of an integer column whose sums stay below 2^53 (same flag in every segment)
// A RESIDUAL leaf: a dictionary leaf of a flat AND that would run on the filter kernel's candidates (DevLeaf::gather) and
// whose column is a field of the row group.  The filter kernel leaves it out and hands its survivors over as candidates;
// this kernel tests the leaf on the row it loads anyway, so a candidate's row is read once instead of twice.
struct DevRowLeaf {
  uint32_t off, bits;       // dictId field of the row
  uint32_t lo, span;        // set == nullptr: match iff (dictId - lo) < span (unsigned)
  const uint32_t* set;      // IN / NOT IN: bitset over dictIds, bit ^ excl
  uint32_t excl, pad;
};
#define PB_ROWS_MAX_LEAVES 4
struct DevRowSeg {
  const uint32_t* rows;
  uint64_t doc_base;
  int32_t table, n_leaves;
  DevRowKey keys[PB_MAX_GROUP_BY];
  DevRowAgg aggs[PB_MAX_AGGS];
  DevRowLeaf leaves[PB_ROWS_MAX_LEAVES];
};
#define PB_ROWS_SMEM_SEGS 16

// field of `bits` bits at bit `off` of a row held in registers (words already byte-swapped, MSB first)
template <int RW>
__device__ __forceinline__ uint32_t pb_row_field(const uint32_t (&w)[RW], uint32_t off, uint32_t bits) {
  const uint32_t wi = off >> 5, sh = off & 31u;
  uint32_t hi = w[0], lo = RW > 1 ? w[1 % RW] : 0u;
#pragma unroll
  for (int k = 1; k < RW; k++) if (wi == (uint32_t)k) { hi = w[k]; lo = k + 1 < RW ? w[(k + 1) % RW] : 0u; }
  return __funnelshift_l(lo, hi, sh) >> (32u - bits);
}

template <int RW>
__global__ void __launch_bounds__(PB_AGG_SMEM_THREADS, 1) pb_agg_rows_kernel(const __grid_constant__ DevQuery Q, const DevRowSeg* __restrict__ gsegs) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  __shared__ DevRowSeg s_segs[PB_ROWS_SMEM_SEGS];
  __shared__ unsigned long long s_doc_base[PB_AGG_MAX_SEGS_SMEM + 1];
  const int tid = threadIdx.x, warp = tid >> 5;
  const int n_segs = Q.n_segs, nG = Q.n_group_by, nA = Q.n_aggs;
  const int n_smem = n_segs < PB_AGG_MAX_SEGS_SMEM ? n_segs : PB_AGG_MAX_SEGS_SMEM;
  for (int i = tid; i < n_smem; i += PB_AGG_SMEM_THREADS) s_doc_base[i] = gsegs[i].doc_base;
  const bool segs_in_smem = n_segs <= PB_ROWS_SMEM_SEGS;
  if (segs_in_smem) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(gsegs);
    uint32_t* dst = reinterpret_cast<uint32_t*>(s_segs);
    for (int i = tid; i < (int)(sizeof(DevRowSeg) / 4) * n_segs; i += PB_AGG_SMEM_THREADS) dst[i] = src[i];
  }
  const DevRowSeg* segs = segs_in_smem ? s_segs : gsegs;
  const unsigned long long n = Q.match_all ? Q.n_docs_total : *Q.match_count;
  // shared-memory table (one table per launch) when it pays
  const uint32_t S = (uint32_t)Q.st_slots, R = (uint32_t)(Q.st_replicas > 0 ? Q.st_replicas : 1);
  SmemTable st;
  st.S = S;
  int n_acc = 0;
  for (int a = 0; a < PB_MAX_AGGS; a++) {
    const int op = a < nA ? Q.agg_op[a] : 0;
    st.acc_of[a] = (a < nA && op >= 1 && op <= 4) ? (int8_t)n_acc++ : (int8_t)-1;
    st.fc_of[a] = -1;
  }
  st.n_fc = 0;
  const size_t rep_bytes = pb_smem_table_bytes(S, 0, n_acc);
  const uint32_t smem0 = pb_smem_u32(smem_raw);
  st.base = smem0 + ((uint32_t)warp & (R - 1)) * (uint32_t)rep_bytes;
  const bool use_smem = S > 0 && n >= Q.st_min_docs;
  if (use_smem) {
    for (uint32_t r = 0; r < R; r++) {
      SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes;
      for (uint32_t i = tid; i < S; i += PB_AGG_SMEM_THREADS) pb_sh_st_u32(z.cnt(i), 0u);
      for (int a = 0; a < nA; a++) {
        if (st.acc_of[a] < 0) continue;
        const unsigned long long init = (Q.agg_op[a] == 1 || Q.agg_op[a] == 4) ? 0ull : 0x7fffffffffffffffull;
        for (uint32_t i = tid; i < S; i += PB_AGG_SMEM_THREADS) pb_sh_st_u64(z.acc(st.acc_of[a], i), init);
      }
    }
  }
  __syncthreads();

  // One doc = one row, fetched with ONE vector load (rows never straddle a 32-byte sector) and taken apart in registers:
  // the aggregation is latency-bound (ncu: 34 warps waiting on memory per issue slot when every field was its own load),
  // so the chain per doc is kept at match list -> row -> remap, and every thread works on two docs at a time.
  auto process = [&](unsigned long long gdoc, const uint32_t (&w)[RW], const DevRowSeg& sg) {
    auto field = [&](uint32_t off, uint32_t bits) -> uint32_t { return pb_row_field<RW>(w, off, bits); };
    uint64_t slot = 0;
    for (int j = 0; j < nG; j++) {
      const DevRowKey& k = sg.keys[j];
      uint32_t id = field(k.off, k.bits);
      if (k.remap) id = (uint32_t)__ldg(k.remap + id);
      slot += (uint64_t)id * k.mult;
    }
    // the row's value field of aggregation a, widened to double like BlockValSet.getDoubleValuesSV
    auto value_of = [&](int a) -> double {
      const DevRowAgg& g = sg.aggs[a];
      const uint32_t w0 = field(g.off, 32u);
      if (g.width == 4) return g.type == 2 ? (double)__uint_as_float(w0) : (double)(int32_t)w0;
      const unsigned long long u = ((unsigned long long)w0 << 32) | field(g.off + 32u, 32u);
      return g.type == 3 ? __longlong_as_double((long long)u) : (double)(long long)u;
    };
    auto ivalue_of = [&](int a) -> long long {           // INT / LONG fields only
      const DevRowAgg& g = sg.aggs[a];
      const uint32_t w0 = field(g.off, 32u);
      if (g.width == 4) return (long long)(int32_t)w0;
      return (long long)(((unsigned long long)w0 << 32) | field(g.off + 32u, 32u));
    };
    if (use_smem) {
      const uint32_t sl = (uint32_t)slot;
      pb_sh_add_u32(st.cnt(sl), 1u);
      for (int a = 0; a < nA; a++) {
        const int op = Q.agg_op[a];
        if (op == 0) continue;
        const double v = ((op == 1 || op == 4) && sg.aggs[a].exact_int) ? 0.0 : value_of(a);
        const uint32_t cell = st.acc(st.acc_of[a], sl);
        if ((op == 1 || op == 4) && sg.aggs[a].exact_int) {
          // exact integer sum: the cell is an int64 kept as two u32 halves, low half first; the carry out of the low half
          // (seen in the value the returning add hands back) rides on the add to the high half -- two native ATOMS, no loop
          const long long iv = ivalue_of(a);
          const uint32_t vlo = (uint32_t)iv, vhi = (uint32_t)((unsigned long long)iv >> 32);
          uint32_t add_hi = vhi;
          if (vlo) { const uint32_t before = pb_sh_atom_add_u32(cell, vlo); add_hi += (before + vlo) < vlo ? 1u : 0u; }
          if (add_hi) pb_sh_add_u32(cell + 4u, add_hi);
        } else if (op == 1 || op == 4) {
          unsigned long long old = pb_sh_ld_u64(cell), assumed;
          do {
            assumed = old;
            old = pb_sh_cas_u64(cell, assumed, (unsigned long long)__double_as_longlong(__longlong_as_double((long long)assumed) + v));
          } while (old != assumed);
        } else if (v == v) {
          const long long e = op == 2 ? pb_enc_f64(v) : ~pb_enc_f64(v);
          long long old = (long long)pb_sh_ld_u64(cell);
          while (e < old) {
            const long long seen = (long long)pb_sh_cas_u64(cell, (unsigned long long)old, (unsigned long long)e);
            if (seen == old) break;
            old = seen;
          }
        }
      }
    } else {
      const DevTable& t = Q.tables[sg.table];
      pb_red_add_u64(&t.rowcnt[slot], 1ull);
      if (t.first_doc) asm volatile("red.global.min.u32 [%0], %1;" ::"l"(t.first_doc + slot), "r"((uint32_t)(gdoc - sg.doc_base)));
      for (int a = 0; a < nA; a++) {
        const int op = Q.agg_op[a];
        if (op == 0) continue;
        const double v = value_of(a);
        if (op == 1 || op == 4) pb_red_add_f64(&t.sum[a][slot], v);
        else if (v == v) pb_red_min_s64(&t.mm[a][slot], op == 2 ? pb_enc_f64(v) : ~pb_enc_f64(v));   // (few matches: a read-before-RED would only add a dependent L2 round trip)
      }
    }
  };
  auto seg_of = [&](unsigned long long gdoc) -> int {
    int lo = 0, hi = n_segs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      const unsigned long long b = mid < PB_AGG_MAX_SEGS_SMEM ? s_doc_base[mid] : gsegs[mid].doc_base;
      if (b <= gdoc) lo = mid; else hi = mid - 1;
    }
    return lo;
  };
  auto load_row = [&](const DevRowSeg& sg, unsigned long long gdoc, uint32_t (&w)[RW]) {
    const uint32_t* __restrict__ row = sg.rows + (gdoc - sg.doc_base) * (unsigned long long)RW;
    if (RW == 2) { const uint2 v = __ldg(reinterpret_cast<const uint2*>(row)); w[0] = v.x; w[1 % RW] = v.y; }
    else {
#pragma unroll
      for (int q4 = 0; q4 < RW / 4; q4++) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(row) + q4);
        w[(4 * q4) % RW] = v.x; w[(4 * q4 + 1) % RW] = v.y; w[(4 * q4 + 2) % RW] = v.z; w[(4 * q4 + 3) % RW] = v.w;
      }
    }
#pragma unroll
    for (int k = 0; k < RW; k++) w[k] = pb_bswap32(w[k]);
  };
  // the residual leaves of the doc's segment against its row: a candidate that fails one is dropped before any table update
  auto passes = [&](const uint32_t (&w)[RW], const DevRowSeg& sg) -> bool {
    for (int k = 0; k < sg.n_leaves; k++) {
      const DevRowLeaf& l = sg.leaves[k];
      const uint32_t id = pb_row_field<RW>(w, l.off, l.bits);
      const bool ok = l.set ? (((__ldg(l.set + (id >> 5)) >> (id & 31)) & 1u) ^ l.excl) != 0u : (id - l.lo) < l.span;
      if (!ok) return false;
    }
    return true;
  };
  // docs_matched (Q.agg_counts_docs): passing docs counted per thread for one table at a time
  int cnt_table = 0;
  uint32_t cnt = 0;
  auto count = [&](int table) {
    if (table != cnt_table && cnt) { pb_red_add_u64(Q.tables[cnt_table].docs_matched, cnt); cnt = 0; }
    cnt_table = table; cnt++;
  };
  const unsigned long long stride = (unsigned long long)gridDim.x * PB_AGG_SMEM_THREADS;
  for (unsigned long long i = (unsigned long long)blockIdx.x * PB_AGG_SMEM_THREADS + tid; i < n; i += 2 * stride) {
    const bool two = i + stride < n;
    const unsigned long long gdoc0 = Q.match_all ? i : (unsigned long long)__ldg(Q.match_list + i);
    const unsigned long long gdoc1 = !two ? gdoc0 : (Q.match_all ? i + stride : (unsigned long long)__ldg(Q.match_list + i + stride));
    const DevRowSeg& sg0 = segs[seg_of(gdoc0)];
    const DevRowSeg& sg1 = segs[seg_of(gdoc1)];
    uint32_t w0[RW], w1[RW];
    load_row(sg0, gdoc0, w0);
    load_row(sg1, gdoc1, w1);
    const bool ok0 = passes(w0, sg0), ok1 = two && passes(w1, sg1);
    if (ok0) process(gdoc0, w0, sg0);
    if (ok1) process(gdoc1, w1, sg1);
    if (Q.agg_counts_docs) { if (ok0) count(sg0.table); if (ok1) count(sg1.table); }
  }
  if (Q.agg_counts_docs) {
    // one reduction per warp when its lanes counted for one table (always so with PB_Q_COMBINE), else one per lane
    const unsigned has = __ballot_sync(0xffffffffu, cnt != 0);
    if (has) {
      const int leader = __ffs(has) - 1;
      const int t0 = __shfl_sync(0xffffffffu, cnt_table, leader);
      if (__all_sync(0xffffffffu, cnt == 0 || cnt_table == t0)) {
        const uint32_t sum = __reduce_add_sync(0xffffffffu, cnt);
        if ((tid & 31) == leader) pb_red_add_u64(Q.tables[t0].docs_matched, sum);
      } else if (cnt) pb_red_add_u64(Q.tables[cnt_table].docs_matched, cnt);
    }
  }
  if (!use_smem) return;
  __syncthreads();
  const DevTable& t = Q.tables[0];
  for (uint32_t i = tid; i < S; i += PB_AGG_SMEM_THREADS) {
    unsigned long long c = 0;
    for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; c += pb_sh_ld_u32(z.cnt(i)); }
    if (c == 0) continue;
    pb_red_add_u64(&t.rowcnt[i], c);
    for (int a = 0; a < nA; a++) {
      if (st.acc_of[a] < 0) continue;
      const int op = Q.agg_op[a];
      if ((op == 1 || op == 4) && segs[0].aggs[a].exact_int) {
        long long v = 0;
        for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; v += (long long)pb_sh_ld_u64(z.acc(st.acc_of[a], i)); }
        pb_red_add_f64(&t.sum[a][i], (double)v);                 // exact: |v| < 2^53
      } else if (op == 1 || op == 4) {
        double v = 0.0;
        for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; v += __longlong_as_double((long long)pb_sh_ld_u64(z.acc(st.acc_of[a], i))); }
        pb_red_add_f64(&t.sum[a][i], v);
      } else {
        long long m = 0x7fffffffffffffffLL;
        for (uint32_t r = 0; r < R; r++) { SmemTable z = st; z.base = smem0 + r * (uint32_t)rep_bytes; const long long o = (long long)pb_sh_ld_u64(z.acc(st.acc_of[a], i)); m = o < m ? o : m; }
        if (m != 0x7fffffffffffffffLL) pb_red_min_s64(&t.mm[a][i], m);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// bitmap-producing kernels (inverted index / sorted index / caller bitmaps -> flat doc bitmaps)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pb_ld_le16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
__device__ __forceinline__ uint32_t pb_ld_le32(const uint8_t* p) { return pb_ld_le16(p) | (pb_ld_le16(p + 2) << 16); }
__device__ __forceinline__ uint32_t pb_ld_be32(const uint8_t* p) {
  return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
}

// One item = one RoaringBitmap of a .bitmap.inv buffer (portable format) OR one list of sorted-index docId ranges, ORed
// into a flat doc bitmap.  All index leaves of all segments of a query are expanded by ONE launch: grid = (32, n_items).
// InvertedIndexFilterOperator.java:60-96 / BitmapInvertedIndexReader.java:45-62 / SortedIndexBasedFilterOperator.java:61-131.
struct DevExpandItem {
  const uint8_t* inv;      // kind 0: the inverted index buffer
  const int32_t* pairs;    // kind 1: inclusive (start,end) docId pairs
  uint32_t* out;           // flat bitmap (bit d&31 of word d>>5)
  int32_t kind;            // 0 = roaring bitmap of dictId `id`, 1 = docId ranges
  int32_t card;
  int32_t id;
  int32_t n_pairs;
  uint32_t num_docs;
  uint32_t pad;
};

static __global__ void pb_expand_kernel(const DevExpandItem* __restrict__ items) {
  const DevExpandItem it = items[blockIdx.y];
  uint32_t* __restrict__ out = it.out;
  if (it.kind == 1) {
    for (int r = blockIdx.x; r < it.n_pairs; r += gridDim.x) {
      uint32_t lo = (uint32_t)it.pairs[2 * r], hi = (uint32_t)it.pairs[2 * r + 1];   // inclusive
      uint32_t w0 = lo >> 5, w1 = hi >> 5;
      for (uint32_t w = w0 + threadIdx.x; w <= w1; w += blockDim.x) {
        uint32_t m = 0xffffffffu;
        if (w == w0) m &= 0xffffffffu << (lo & 31);
        if (w == w1) m &= 0xffffffffu >> (31 - (hi & 31));
        atomicOr(&out[w], m);
      }
    }
    return;
  }
  const uint8_t* inv = it.inv;
  const uint32_t num_docs = it.num_docs;
  const uint32_t first = pb_ld_be32(inv);
  const uint32_t s = pb_ld_be32(inv + 4ull * it.id), e = pb_ld_be32(inv + 4ull * it.id + 4);
  const uint8_t* blob = inv + 4ull * ((uint64_t)it.card + 1) + (s - first);
  if (e - s < 8) return;
  const uint32_t cookie = pb_ld_le32(blob);
  uint32_t n, p;
  const uint8_t* run_bitmap = nullptr;
  bool has_offsets;
  if ((cookie & 0xffffu) == 12347u) { n = (cookie >> 16) + 1; run_bitmap = blob + 4; p = 4 + (n + 7) / 8; has_offsets = n >= 4; }
  else if (cookie == 12346u) { n = pb_ld_le32(blob + 4); p = 8; has_offsets = true; }
  else return;
  const uint8_t* hdr = blob + p;
  const uint8_t* offs = hdr + 4ull * n;
  const uint32_t data0 = p + 4 * n + (has_offsets ? 4 * n : 0);
  for (uint32_t c = blockIdx.x; c < n; c += gridDim.x) {
    uint32_t key = pb_ld_le16(hdr + 4 * c), ccard = pb_ld_le16(hdr + 4 * c + 2) + 1;
    bool is_run = run_bitmap && ((run_bitmap[c >> 3] >> (c & 7)) & 1);
    uint32_t off;
    if (has_offsets) off = pb_ld_le32(offs + 4 * c);
    else {   // < 4 containers, no offset header: walk the sizes
      off = data0;
      for (uint32_t k = 0; k < c; k++) {
        uint32_t kc = pb_ld_le16(hdr + 4 * k + 2) + 1;
        bool kr = run_bitmap && ((run_bitmap[k >> 3] >> (k & 7)) & 1);
        off += kr ? 2 + 4 * pb_ld_le16(blob + off) : (kc <= 4096 ? 2 * kc : 8192);
      }
    }
    const uint8_t* d = blob + off;
    const uint32_t base = key << 16;
    if (is_run) {
      uint32_t nr = pb_ld_le16(d);
      for (uint32_t r = 0; r < nr; r++) {
        uint32_t st = pb_ld_le16(d + 2 + 4 * r), len = pb_ld_le16(d + 4 + 4 * r);
        for (uint32_t k = threadIdx.x; k <= len; k += blockDim.x) {
          uint32_t doc = base | (st + k);
          if (doc < num_docs) atomicOr(&out[doc >> 5], 1u << (doc & 31));
        }
      }
    } else if (ccard <= 4096) {
      for (uint32_t k = threadIdx.x; k < ccard; k += blockDim.x) {
        uint32_t doc = base | pb_ld_le16(d + 2 * k);
        if (doc < num_docs) atomicOr(&out[doc >> 5], 1u << (doc & 31));
      }
    } else {
      for (uint32_t k = threadIdx.x; k < 2048; k += blockDim.x) {
        uint32_t w = pb_ld_le32(d + 4 * k);
        uint32_t wi = (base >> 5) + k;
        if (w && (uint64_t)wi * 32 < num_docs) atomicOr(&out[wi], w);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// table init / finalize
// ------------------------------------------------------------------------------------------------
// one launch initialises every table of the query: zero region (row counts, sums, distinct bitsets, counters),
// 0xFF region (hash keys = PB_HASH_EMPTY) and the min/max region (INT64_MAX: larger than any encoded value)
// The first head_n16 16-byte words of the zero region are the per-table counter cells: they start from the host-known
// values in `head` (total docs, entries scanned in filter, docs matched of a match-all query) instead of zero, so that a
// cross-GPU merge sums them like every other counter.  `aux` is a second zero region (per-wave match counters and
// per-segment swim-lane statistics) that is not part of the merged block.
static __global__ void pb_init_tables_kernel(uint4* zero, uint64_t zero_n16, uint4* ff, uint64_t ff_n16, uint4* mm, uint64_t mm_n16,
                                      uint4* aux, uint64_t aux_n16, const uint4* __restrict__ head, uint64_t head_n16,
                                      const unsigned int* only_if = nullptr) {
  if (only_if && *only_if == 0) return;      // (the conditional re-initialisation of a repair pass)
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x, t0 = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint4 z = make_uint4(0u, 0u, 0u, 0u), f = make_uint4(~0u, ~0u, ~0u, ~0u), m = make_uint4(~0u, 0x7fffffffu, ~0u, 0x7fffffffu);
  for (uint64_t i = t0; i < zero_n16; i += stride) zero[i] = i < head_n16 ? head[i] : z;
  for (uint64_t i = t0; i < ff_n16; i += stride) ff[i] = f;
  for (uint64_t i = t0; i < mm_n16; i += stride) mm[i] = m;
  for (uint64_t i = t0; i < aux_n16; i += stride) aux[i] = z;
}

// Filtered aggregations: ExecutionStatistics of the swim-lanes (FilteredGroupByOperator.java:146-149), reduced from the
// per-segment counters to two cells of the segment's table so that they merge across GPUs with the other counters.
// Per segment and lane l (0 = the non-filtered lane, 1 + f = FILTER clause f): docs_w = 1 when the lane's docs count
// towards numDocsScanned, post_w = the lane's projected columns (numEntriesScannedPostFilter = docs x columns).
struct DevLaneWeights { int32_t table; int32_t docs_w[1 + PB_MAX_AGG_FILTERS]; int32_t post_w[1 + PB_MAX_AGG_FILTERS]; int32_t pad; };
static __global__ void pb_lane_stats_kernel(const DevLaneWeights* __restrict__ w, const unsigned long long* __restrict__ seg_stats, int n_segs,
                                     int n_lanes, unsigned long long* counters, int cells_per_table) {
  for (int si = blockIdx.x * blockDim.x + threadIdx.x; si < n_segs; si += gridDim.x * blockDim.x) {
    const unsigned long long* ss = seg_stats + (size_t)si * (1 + PB_MAX_AGG_FILTERS);
    unsigned long long docs = 0, post = 0;
    for (int l = 0; l < n_lanes; l++) { docs += ss[l] * (unsigned long long)w[si].docs_w[l]; post += ss[l] * (unsigned long long)w[si].post_w[l]; }
    unsigned long long* c = counters + (size_t)w[si].table * cells_per_table;
    if (docs) atomicAdd(c + 4, docs);
    if (post) atomicAdd(c + 5, post);
  }
}

// cross-GPU merge: reduce n_rows copies of the table block element-wise into `dst` with the operator of each region:
// counters + row counts u64 SUM | sums f64 SUM | distinct bitsets OR | min/max i64 MIN.  The copies are either the rows of one
// buffer (`gathered`, row-major: the receive buffer of an all-gather, which includes this rank's own block) or, when
// `peers` is set, blocks read in place from the peer GPUs over NVLink (one process driving several devices); with
// base_is_dst the copy already in `dst` is the first operand.  Sums are added in row order, so every rank computes the same
// bits from the same gathered buffer.
#define PB_MERGE_MAX_PEERS 16
struct DevMergePeers { const unsigned long long* p[PB_MERGE_MAX_PEERS]; };
static __global__ void pb_merge_blocks_kernel(unsigned long long* __restrict__ dst, const unsigned long long* __restrict__ gathered, const DevMergePeers peers,
                                       int n_rows, int base_is_dst, uint64_t n_words, uint64_t sum_off, uint64_t dc_off, uint64_t mm_off) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_words; i += (uint64_t)gridDim.x * blockDim.x) {
    auto row = [&](int r) -> unsigned long long { return gathered ? gathered[(uint64_t)r * n_words + i] : peers.p[r][i]; };
    unsigned long long v = base_is_dst ? dst[i] : row(0);
    const int r0 = base_is_dst ? 0 : 1;
    if (i < sum_off) { for (int r = r0; r < n_rows; r++) v += row(r); }
    else if (i < dc_off) { double d = __longlong_as_double((long long)v); for (int r = r0; r < n_rows; r++) d += __longlong_as_double((long long)row(r)); v = (unsigned long long)__double_as_longlong(d); }
    else if (i < mm_off) { for (int r = r0; r < n_rows; r++) v |= row(r); }
    else { long long m = (long long)v; for (int r = r0; r < n_rows; r++) { long long o = (long long)row(r); m = o < m ? o : m; } v = (unsigned long long)m; }
    dst[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// hash tables across ranks (SURVEY.md §8e: "partition tuples by hash(key) % nGPU, one all-to-all, local merge kernel"; the
// reference merges by key in IndexedTable.upsert, CTR/data/table/IndexedTable.java:99-125).  A tuple is
// [key words | row count | one u64 per aggregation (f64 sum bits / encoded min-max / filtered row count)].
// ------------------------------------------------------------------------------------------------
struct DevHashXfer {
  int32_t n_ranks, key_words, n_aggs, tuple_words;
  uint64_t S;                                   // slots to scan (capacity + the sentinel slot)
  uint64_t capacity;
  const unsigned long long* hkeys;
  const unsigned long long* rowcnt;
  const double* sum[PB_MAX_AGGS];
  const long long* mm[PB_MAX_AGGS];
  const unsigned long long* fcnt[PB_MAX_AGGS];
  unsigned long long* counts;                   // [n_ranks] tuples per destination
  unsigned long long* cursors;                  // [n_ranks] running positions while packing
  const unsigned long long* offsets;            // [n_ranks] first tuple of each destination in `out`
  unsigned long long* out;                      // packed tuples, grouped by destination
};
__device__ __forceinline__ uint32_t pb_owner_rank(unsigned long long klo, unsigned long long khi, int key_words, int n_ranks) {
  // a different mix than the slot hash, so that a rank's partition still spreads over its whole table
  unsigned long long h = pb_hash64((key_words == 2 ? (klo ^ pb_hash64(khi)) : klo) ^ 0x9e3779b97f4a7c15ull);
  return (uint32_t)((h >> 32) % (unsigned)n_ranks);
}
__device__ __forceinline__ void pb_slot_key(const DevHashXfer& X, uint64_t i, unsigned long long& klo, unsigned long long& khi) {
  if (X.key_words == 2) { klo = i == X.capacity ? PB_HASH_EMPTY : X.hkeys[2 * i]; khi = i == X.capacity ? PB_HASH_EMPTY : X.hkeys[2 * i + 1]; }
  else { klo = i == X.capacity ? PB_HASH_EMPTY : X.hkeys[i]; khi = 0; }
}
static __global__ void pb_hash_count_kernel(const DevHashXfer X) {
  __shared__ unsigned int s_cnt[64];
  for (int k = threadIdx.x; k < X.n_ranks; k += blockDim.x) s_cnt[k] = 0;
  __syncthreads();
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < X.S; i += (uint64_t)gridDim.x * blockDim.x) {
    if (X.rowcnt[i] == 0) continue;
    unsigned long long klo, khi;
    pb_slot_key(X, i, klo, khi);
    atomicAdd(&s_cnt[pb_owner_rank(klo, khi, X.key_words, X.n_ranks)], 1u);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < X.n_ranks; k += blockDim.x) if (s_cnt[k]) atomicAdd(&X.counts[k], (unsigned long long)s_cnt[k]);
}
static __global__ void pb_hash_pack_kernel(const DevHashXfer X) {
  const int lane = threadIdx.x & 31;
  const uint64_t S_round = (X.S + 31) & ~(uint64_t)31;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < S_round; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long c = i < X.S ? X.rowcnt[i] : 0ull;
    unsigned long long klo = 0, khi = 0;
    uint32_t dest = 0xffffffffu;
    if (c) { pb_slot_key(X, i, klo, khi); dest = pb_owner_rank(klo, khi, X.key_words, X.n_ranks); }
    // lanes bound for the same destination share one atomic
    const unsigned peers = __match_any_sync(0xffffffffu, dest);
    if (!c) continue;
    const int leader = __ffs(peers) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(&X.cursors[dest], (unsigned long long)__popc(peers));
    base = __shfl_sync(peers, base, leader);
    unsigned long long* o = X.out + (X.offsets[dest] + base + __popc(peers & ((1u << lane) - 1u))) * (uint64_t)X.tuple_words;
    int w = 0;
    o[w++] = klo;
    if (X.key_words == 2) o[w++] = khi;
    o[w++] = c;
    for (int a = 0; a < X.n_aggs; a++)
      o[w++] = X.sum[a] ? (unsigned long long)__double_as_longlong(X.sum[a][i]) : X.mm[a] ? (unsigned long long)X.mm[a][i] : X.fcnt[a] ? X.fcnt[a][i] : 0ull;
  }
}
// received tuples -> this rank's (re-initialised) table
static __global__ void pb_hash_merge_kernel(const DevTable t, const unsigned long long* __restrict__ in, uint64_t n_tuples, int key_words, int n_aggs, int tuple_words) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_tuples; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long* p = in + i * (uint64_t)tuple_words;
    int w = 0;
    const unsigned long long klo = p[w++];
    const unsigned long long khi = key_words == 2 ? p[w++] : 0ull;
    const unsigned long long c = p[w++];
    const uint64_t slot = key_words == 2 ? pb_hash_slot2(t, klo, khi) : pb_hash_slot(t, klo);
    if (slot == ~0ull) continue;                 // numGroupsLimit of the merged table (IndexedTable drops new keys past its limit too)
    pb_red_add_u64(&t.rowcnt[slot], c);
    for (int a = 0; a < n_aggs; a++) {
      const unsigned long long v = p[w++];
      if (t.sum[a]) pb_red_add_f64(&t.sum[a][slot], __longlong_as_double((long long)v));
      else if (t.mm[a]) pb_red_min_s64(&t.mm[a][slot], (long long)v);
      else if (t.fcnt[a]) pb_red_add_u64(&t.fcnt[a][slot], v);
    }
  }
}
// counter cells of all ranks (rank-major) summed into this rank's; the group count [0] and the cursor [3] stay local
static __global__ void pb_sum_counters_kernel(unsigned long long* cells, const unsigned long long* __restrict__ gathered, int n_ranks, int n_cells) {
  const int i = threadIdx.x;
  if (i >= n_cells || i == 0 || i == 3) return;
  unsigned long long v = 0;
  for (int r = 0; r < n_ranks; r++) v += gathered[r * n_cells + i];
  cells[i] = v;
}

// numGroupsLimit in doc order: *thr = the limit-th smallest first_doc among the existing groups (first docs are distinct: a
// doc belongs to one group), or 0xFFFFFFFE when fewer groups exist.  One CTA, four 8-bit radix-select passes.
static __global__ void pb_select_first_kernel(const uint32_t* __restrict__ first_doc, uint64_t S, uint32_t limit, uint32_t* thr) {
  __shared__ unsigned int hist[256];
  __shared__ uint32_t s_prefix, s_k, s_done;
  if (threadIdx.x == 0) { s_prefix = 0; s_k = limit; s_done = 0; }
  __syncthreads();
  for (int pass = 3; pass >= 0; pass--) {
    for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
    __syncthreads();
    const uint32_t prefix = s_prefix, hi_mask = pass == 3 ? 0u : (0xffffffffu << (8 * (pass + 1)));
    for (uint64_t i = threadIdx.x; i < S; i += blockDim.x) {
      const uint32_t v = first_doc[i];
      if (v != 0xffffffffu && (v & hi_mask) == (prefix & hi_mask)) atomicAdd(&hist[(v >> (8 * pass)) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t k = s_k, cum = 0;
      int b = 0;
      for (; b < 256; b++) { if (cum + hist[b] >= k) break; cum += hist[b]; }
      if (b == 256) s_done = 1;                       // fewer than `limit` groups exist: everything survives
      else { s_prefix = prefix | ((uint32_t)b << (8 * pass)); s_k = k - cum; }
    }
    __syncthreads();
    if (s_done) break;
  }
  if (threadIdx.x == 0) *thr = s_done ? 0xfffffffeu : s_prefix;
}

// DISTINCTCOUNT on raw columns: distinct values per slot, from the table-wide (slot, value) set
static __global__ void pb_dset_count_kernel(const unsigned long long* __restrict__ keys, uint64_t cap, unsigned long long* __restrict__ dcnt) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long slot = keys[2 * i];
    if (slot != PB_HASH_EMPTY || keys[2 * i + 1] != PB_HASH_EMPTY) atomicAdd(&dcnt[slot], 1ull);
  }
}
// ... and the value sets themselves: the values of compacted group k land (unordered) at out[offsets[k] ..)
static __global__ void pb_dset_scatter_kernel(const unsigned long long* __restrict__ keys, uint64_t cap, const uint32_t* __restrict__ group_of_slot,
                                              const unsigned long long* __restrict__ offsets, unsigned long long* cursors, long long* __restrict__ out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < cap; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long slot = keys[2 * i], v = keys[2 * i + 1];
    if (slot == PB_HASH_EMPTY && v == PB_HASH_EMPTY) continue;
    const uint32_t k = group_of_slot[slot];
    if (k == 0xffffffffu) continue;
    out[offsets[k] + atomicAdd(&cursors[k], 1ull)] = (long long)v;
  }
}
static __global__ void pb_invert_slots_kernel(const unsigned long long* __restrict__ slots, uint64_t n, uint32_t* __restrict__ group_of_slot) {
  for (uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) group_of_slot[slots[k]] = (uint32_t)k;
}

// ------------------------------------------------------------------------------------------------
// ORDER BY ... LIMIT trim of a group table (the server-side trim of the combine layer: IndexedTable + TableResizer keep
// max(5 x LIMIT, minServerGroupTrimSize) groups once a table passes groupTrimThreshold: CTR/util/GroupByUtils.java:44-70,
// CTR/data/table/TableResizer.java).  okey[slot] = the first ORDER BY expression as an unsigned 64-bit rank (larger = earlier
// in the requested order); a grid-wide radix select finds the trim_size-th largest; the hand-back emits the groups at or
// above it (ties at the boundary are all kept: the broker's final sort decides among them).
// ------------------------------------------------------------------------------------------------
struct DevOrderKey {
  int32_t kind;              // 0 = group-by column, 1 = aggregation
  int32_t descending;
  int32_t mode, key_words;   // table mode / hash key words
  int32_t op;                // aggregation: PB_AGG_*
  int32_t field_is_signed;   // group column: raw INT / LONG value (signed order)
  int32_t field_is_double;   // group column: raw FLOAT / DOUBLE value (bits of the double)
  int32_t shift, width;      // hash: field position
  uint64_t div, card;        // dense: field = (slot / div) % card
  uint64_t S, capacity;
  const unsigned long long* rowcnt;
  const unsigned long long* hkeys;
  const double* sum;
  const long long* mm;
  const unsigned long long* fcnt;
  unsigned long long* okey;
};
static __global__ void pb_order_key_kernel(const DevOrderKey K) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < K.S; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long c = K.rowcnt[i];
    unsigned long long u = 0;
    if (c) {
      if (K.kind == 1) {
        long long e;
        if (K.op == 0) e = (long long)(K.fcnt ? K.fcnt[i] : c);                                        // COUNT
        else if (K.op == 1) e = pb_enc_f64(K.sum[i]);                                                   // SUM
        else if (K.op == 4) { const unsigned long long n = K.fcnt ? K.fcnt[i] : c; e = pb_enc_f64(n ? K.sum[i] / (double)n : 0.0); }   // AVG
        else e = K.op == 2 ? K.mm[i] : ~K.mm[i];                                                        // MIN / MAX (encoded; MAX is stored complemented)
        u = (unsigned long long)e ^ 0x8000000000000000ull;
      } else {
        uint64_t field;
        if (K.mode == T_DENSE) field = (i / K.div) % K.card;
        else {
          unsigned long long klo, khi = 0;
          if (K.key_words == 2) { klo = i == K.capacity ? PB_HASH_EMPTY : K.hkeys[2 * i]; khi = i == K.capacity ? PB_HASH_EMPTY : K.hkeys[2 * i + 1]; }
          else klo = i == K.capacity ? PB_HASH_EMPTY : K.hkeys[i];
          if (K.shift < 64) { field = klo >> K.shift; if (K.shift && K.shift + K.width > 64) field |= khi << (64 - K.shift); }
          else field = khi >> (K.shift - 64);
          if (K.width < 64) field &= ((1ull << K.width) - 1ull);
        }
        if (K.field_is_double) u = (unsigned long long)pb_enc_f64(__longlong_as_double((long long)field)) ^ 0x8000000000000000ull;
        else if (K.field_is_signed) u = (K.width == 32 ? (unsigned long long)(long long)(int32_t)(uint32_t)field : field) ^ 0x8000000000000000ull;
        else u = field;                                                                                  // dictId: sorted dictionary order
      }
      if (!K.descending) u = ~u;
    }
    K.okey[i] = u;
  }
}
// radix select, one 8-bit digit per pass: state = {prefix, k remaining, done, threshold, candidates}
struct DevSelectState { unsigned long long prefix, k, done, thr, total; unsigned long long hist[256]; };
static __global__ void pb_rselect_hist_kernel(const unsigned long long* __restrict__ okey, const unsigned long long* __restrict__ rowcnt, uint64_t S, int pass,
                                              DevSelectState* st) {
  __shared__ unsigned int h[256];
  for (int b = threadIdx.x; b < 256; b += blockDim.x) h[b] = 0;
  __syncthreads();
  if (!st->done) {
    const unsigned long long prefix = st->prefix;
    const unsigned long long hi_mask = pass == 7 ? 0ull : (~0ull << (8 * (pass + 1)));
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < S; i += (uint64_t)gridDim.x * blockDim.x) {
      if (!rowcnt[i]) continue;
      const unsigned long long v = okey[i];
      if ((v & hi_mask) == (prefix & hi_mask)) atomicAdd(&h[(v >> (8 * pass)) & 255u], 1u);
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < 256; b += blockDim.x) if (h[b]) atomicAdd(&st->hist[b], (unsigned long long)h[b]);
}
static __global__ void pb_rselect_pick_kernel(DevSelectState* st, int pass, unsigned long long trim_size, unsigned long long trim_threshold) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (pass == 7) { st->prefix = 0; st->k = trim_size; st->done = 0; st->thr = 0; }
  if (!st->done) {
    if (pass == 7) {
      unsigned long long total = 0;
      for (int b = 0; b < 256; b++) total += st->hist[b];
      st->total = total;
      if (total <= trim_threshold || total <= st->k) { st->done = 1; st->thr = 0; }      // the table is small enough: keep everything
    }
    if (!st->done) {
      unsigned long long k = st->k, cum = 0;
      int b = 255;
      for (; b >= 0; b--) { if (cum + st->hist[b] >= k) break; cum += st->hist[b]; }      // k-th LARGEST
      if (b < 0) { st->done = 1; st->thr = 0; }
      else { st->prefix |= (unsigned long long)b << (8 * pass); st->k = k - cum; if (pass == 0) st->thr = st->prefix; }
    }
  }
  for (int b = 0; b < 256; b++) st->hist[b] = 0;
}

// count non-empty slots (that survive the ORDER BY trim, if any)
static __global__ void pb_count_groups_kernel(const unsigned long long* __restrict__ rowcnt, uint64_t n, unsigned long long* out,
                                              const unsigned long long* __restrict__ okey, const unsigned long long* __restrict__ othr) {
  unsigned long long c = 0;
  const unsigned long long thr = othr ? *othr : 0ull;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) c += rowcnt[i] != 0 && (!okey || okey[i] >= thr);
  for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// Result hand-back in one pass: compaction of the non-empty groups, aggregate extraction, and group-key decode
// (DictionaryBasedGroupKeyGenerator.getKeys: rawKey -> dictIds -> dictionary values, :578-591) straight into
// page-locked host memory.  Warp-aggregated cursor => each warp writes consecutive rows (coalesced PCIe writes).
struct DevFinKey {
  const uint8_t* dict_vals;   // native-endian dictionary entries on the device (dictionary key columns)
  int32_t eb;                 // bytes per decoded value
  int32_t is_dict;
  int32_t type;               // PB_INT .. PB_STRING
  int32_t shift, width;       // T_HASH: field position in the composite key
  int32_t pad;
  uint64_t div, card;         // T_DENSE: field = (slot / div) % card
  int32_t* out_ids;
  uint8_t* out_vals;
};
struct DevFinAgg {
  int32_t op, pad;
  const double* sum;
  const long long* mm;
  const unsigned long long* fcnt;   // COUNT / AVG with a FILTER clause: row count of the function (else the group's)
  const unsigned long long* dcnt;   // DISTINCTCOUNT on a raw column: distinct values per slot
  double* out;
  long long* out_cnt;               // where fcnt goes (the aggregation's long array)
};
struct DevFinalize {
  int32_t mode, n_gb, n_aggs, always_emit;
  uint64_t S;                 // slots to scan
  int32_t key_words, count_all;   // count_all (PB_Q_NULL_HANDLING): every aggregation's long array carries its row count
  uint64_t capacity;          // T_HASH: index of the reserved sentinel slot
  uint64_t cap_out;
  const unsigned long long* rowcnt;
  const unsigned long long* hkeys;
  const uint32_t* first_doc;      // numGroupsLimit in doc order: emit only groups whose first doc is <= *first_thr
  const uint32_t* first_thr;
  const unsigned long long* okey; // ORDER BY ... LIMIT trim: emit only groups whose order key is >= *othr
  const unsigned long long* othr;
  unsigned long long* cursor;
  unsigned long long* out_slots;
  unsigned long long* out_rows;
  DevFinKey keys[PB_MAX_GROUP_BY];
  DevFinAgg aggs[PB_MAX_AGGS];
};

static __global__ void pb_finalize_kernel(const DevFinalize F) {
  const int lane = threadIdx.x & 31;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t S_round = (F.S + 31) & ~(uint64_t)31;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < S_round; i += stride) {
    const unsigned long long c = i < F.S ? F.rowcnt[i] : 0ull;
    bool emit = i < F.S && (c != 0 || F.always_emit);
    if (emit && F.first_doc && F.first_doc[i] > *F.first_thr) emit = false;
    if (emit && F.okey && F.okey[i] < *F.othr) emit = false;
    const uint32_t b = __ballot_sync(0xffffffffu, emit);
    if (!b) continue;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(F.cursor, (unsigned long long)__popc(b));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (!emit) continue;
    const uint64_t k = base + __popc(b & ((1u << lane) - 1u));
    if (k >= F.cap_out) continue;
    if (F.out_slots) F.out_slots[k] = i;          // (only DISTINCTCOUNT hand-back needs the slot of a row)
    F.out_rows[k] = c;
    for (int a = 0; a < F.n_aggs; a++) {
      const DevFinAgg& fa = F.aggs[a];
      if (fa.sum) fa.out[k] = fa.sum[i];
      else if (fa.mm) {
        // empty group (keyless query without matches): MIN = +inf, MAX = -inf (MinAggregationFunction.java:37 defaults)
        // (same for a group none of whose docs passes the function's FILTER clause: the cell still holds the init pattern)
        if (c == 0 || fa.mm[i] == 0x7fffffffffffffffLL) fa.out[k] = fa.op == 2 ? __longlong_as_double(0x7ff0000000000000LL) : __longlong_as_double((long long)0xfff0000000000000ULL);
        else fa.out[k] = pb_dec_f64(fa.op == 2 ? fa.mm[i] : ~fa.mm[i]);
      }
      else if (fa.op == 0) fa.out[k] = fa.fcnt ? (double)fa.fcnt[i] : (double)c;
      // the aggregation's long array: COUNT value / AVG denominator (the function's own row count under a FILTER clause), 0 otherwise
      if (fa.op == 5 && fa.dcnt) fa.out_cnt[k] = (long long)fa.dcnt[i];
      if (fa.op != 5 && fa.out_cnt) fa.out_cnt[k] = (fa.op == 0 || fa.op == 4 || F.count_all) ? (fa.fcnt ? (long long)fa.fcnt[i] : (long long)c) : 0ll;
    }
    unsigned long long key = 0, key_hi = 0;
    if (F.mode == T_HASH) {
      if (F.key_words == 2) { key = (i == F.capacity) ? PB_HASH_EMPTY : F.hkeys[2 * i]; key_hi = (i == F.capacity) ? PB_HASH_EMPTY : F.hkeys[2 * i + 1]; }
      else key = (i == F.capacity) ? PB_HASH_EMPTY : F.hkeys[i];
    }
    for (int j = 0; j < F.n_gb; j++) {
      const DevFinKey& fk = F.keys[j];
      uint64_t field;
      if (F.mode == T_DENSE) field = (i / fk.div) % fk.card;
      else {
        if (fk.shift < 64) { field = key >> fk.shift; if (fk.shift && fk.shift + fk.width > 64) field |= key_hi << (64 - fk.shift); }
        else field = key_hi >> (fk.shift - 64);
        if (fk.width < 64) field &= ((1ull << fk.width) - 1ull);
      }
      uint8_t* o = fk.out_vals + k * (uint64_t)fk.eb;
      if (fk.is_dict) {
        fk.out_ids[k] = (int32_t)field;
        const uint8_t* src = fk.dict_vals + field * (uint64_t)fk.eb;
        if (fk.eb == 4) *reinterpret_cast<uint32_t*>(o) = *reinterpret_cast<const uint32_t*>(src);
        else if (fk.eb == 8) *reinterpret_cast<unsigned long long*>(o) = *reinterpret_cast<const unsigned long long*>(src);
        else for (int q = 0; q < fk.eb; q++) o[q] = src[q];
      } else {
        fk.out_ids[k] = -1;
        if (fk.type == 0) *reinterpret_cast<int32_t*>(o) = (int32_t)(uint32_t)field;
        else if (fk.type == 2) *reinterpret_cast<float*>(o) = (float)__longlong_as_double((long long)field);
        else *reinterpret_cast<unsigned long long*>(o) = field;
      }
    }
  }
}

// gather kernels used by the two-pass path of very large tables
static __global__ void pb_gather_u64_kernel(const unsigned long long* __restrict__ src, const unsigned long long* __restrict__ slots, uint64_t n, unsigned long long* __restrict__ dst) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) dst[i] = src[slots[i]];
}
// DISTINCTCOUNT: one warp per compacted group: popcount of its bitset
static __global__ void pb_distinct_count_kernel(const uint32_t* __restrict__ bits, uint64_t words, const unsigned long long* __restrict__ slots,
                                         uint64_t n, unsigned long long* __restrict__ out) {
  uint64_t g = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (g >= n) return;
  const uint32_t* b = bits + slots[g] * words;
  unsigned long long c = 0;
  for (uint64_t w = lane; w < words; w += 32) c += __popc(b[w]);
  for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
  if (lane == 0) out[g] = c;
}
// DISTINCTCOUNT value sets: one warp per group writes the ascending dictIds at offsets[g]
static __global__ void pb_distinct_ids_kernel(const uint32_t* __restrict__ bits, uint64_t words, const unsigned long long* __restrict__ slots,
                                       uint64_t n, const unsigned long long* __restrict__ offsets, int32_t* __restrict__ out) {
  uint64_t g = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (g >= n) return;
  const uint32_t* b = bits + slots[g] * words;
  unsigned long long pos = offsets[g];
  for (uint64_t w0 = 0; w0 < words; w0 += 32) {
    uint32_t x = (w0 + lane < words) ? b[w0 + lane] : 0u;
    uint32_t c = __popc(x);
    uint32_t incl = c;
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    unsigned long long my = pos + incl - c;
    while (x) { int bpos = __ffs(x) - 1; x &= x - 1; out[my++] = (int32_t)((w0 + lane) * 32 + bpos); }
    pos += __shfl_sync(0xffffffffu, incl, 31);
  }
}

// Row group build: one thread per doc packs the doc's dictIds of the member columns MSB-first into one row of
// stride_words 32-bit words, in the same big-endian bit order as Pinot's own forward indexes, so that pb_unpack_at_bounded
// reads a field of a row exactly like a value of a column (stride_bits = row stride, bit_off = field offset).
#define PB_ROW_MAX_COLS 16
#define PB_ROW_MAX_WORDS 8
struct DevRowBuild {
  int32_t n_cols, stride_words;
  uint32_t num_docs, pad;
  const uint8_t* fwd[PB_ROW_MAX_COLS];
  const uint8_t* dict_native[PB_ROW_MAX_COLS];   // non-null: the field holds the DECODED dictionary value (value_bytes = 4 or 8), not the dictId
  int32_t value_bytes[PB_ROW_MAX_COLS];
  int32_t bits[PB_ROW_MAX_COLS];
  int32_t bit_off[PB_ROW_MAX_COLS];
  uint32_t* out;
};
static __global__ void pb_build_rows_kernel(const DevRowBuild B) {
  for (uint64_t doc = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; doc < B.num_docs; doc += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t w[PB_ROW_MAX_WORDS];
#pragma unroll
    for (int k = 0; k < PB_ROW_MAX_WORDS; k++) w[k] = 0;
    for (int c = 0; c < B.n_cols; c++) {
      const uint32_t id = pb_unpack_at(B.fwd[c], (uint32_t)doc, B.bits[c]);
      if (B.dict_native[c]) {
        // decoded value, stored like a raw forward index entry (big-endian once the words are swapped below): aggregation
        // inputs then need no dictionary lookup per matching row (a dependent random L2 access each)
        const int k0 = B.bit_off[c] >> 5;
        uint32_t v0, v1 = 0;
        if (B.value_bytes[c] == 4) v0 = reinterpret_cast<const uint32_t*>(B.dict_native[c])[id];
        else { const unsigned long long v = reinterpret_cast<const unsigned long long*>(B.dict_native[c])[id]; v0 = (uint32_t)(v >> 32); v1 = (uint32_t)v; }
#pragma unroll
        for (int kk = 0; kk < PB_ROW_MAX_WORDS; kk++) {
          if (kk == k0) w[kk] = v0;
          if (kk == k0 + 1 && B.value_bytes[c] == 8) w[kk] = v1;
        }
        continue;
      }
      const int p = B.bit_off[c], k = p >> 5, sft = 32 - B.bits[c] - (p & 31);      // left shift that puts the value's LSB in place
#pragma unroll
      for (int kk = 0; kk < PB_ROW_MAX_WORDS; kk++) {
        if (kk == k) w[kk] |= sft >= 0 ? (id << sft) : (id >> (-sft));
        if (kk == k + 1 && sft < 0) w[kk] |= id << (32 + sft);
      }
    }
    uint32_t* o = B.out + doc * (uint64_t)B.stride_words;
#pragma unroll
    for (int k = 0; k < PB_ROW_MAX_WORDS; k++) if (k < B.stride_words) o[k] = pb_bswap32(w[k]);
  }
}

// ------------------------------------------------------------------------------------------------
// Chunk-compressed raw forward indexes (BaseChunkForwardIndexReader.decompressChunk,
// SEGL/segment/index/readers/forward/BaseChunkForwardIndexReader.java:120-160; codecs SEGL/io/compression/LZ4Decompressor.java,
// LZ4WithLengthDecompressor.java, SnappyDecompressor.java): decoded ONCE, at stage time, into the PASS_THROUGH value area the
// scan / gather kernels read -- the compressed bytes are what crosses PCIe.  One warp per chunk: every lane parses the
// sequence headers (uniform loads), the warp copies the literal and match bytes cooperatively.  A match may overlap its own
// output (offset < length = a repeating pattern): byte i of it is byte (i mod offset) of the `offset` bytes before the match,
// all written by earlier sequences.  Every read and write is bounds-checked; a malformed stream sets *err and stops the chunk.
// ------------------------------------------------------------------------------------------------
#define PB_CODEC_SNAPPY 1
#define PB_CODEC_LZ4 3
#define PB_CODEC_LZ4_LENGTH_PREFIXED 4
struct DevChunkDecode {
  const uint8_t* src;          // the compressed chunks, back to back as in the file
  const uint64_t* offs;        // n_chunks + 1 offsets into src
  uint8_t* dst;                // value area: chunk k at k * chunk_bytes
  uint64_t total_bytes;        // num_docs x width (the last chunk is shorter)
  uint32_t n_chunks, chunk_bytes;
  int32_t codec;
  uint32_t* err;
};
static __global__ void __launch_bounds__(256) pb_chunk_decode_kernel(const DevChunkDecode D) {
  const int lane = threadIdx.x & 31;
  const uint32_t chunk = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (chunk >= D.n_chunks) return;
  const uint8_t* in = D.src + D.offs[chunk];
  const uint64_t in_len = D.offs[chunk + 1] - D.offs[chunk];
  uint8_t* out = D.dst + (uint64_t)chunk * D.chunk_bytes;
  const uint64_t left = D.total_bytes - (uint64_t)chunk * D.chunk_bytes;
  const uint64_t out_len = left < D.chunk_bytes ? left : D.chunk_bytes;
  uint64_t ip = 0, op = 0;
  bool bad = false;
  auto copy_literals = [&](uint64_t n) {
    if (ip + n > in_len || op + n > out_len) { bad = true; return; }
    for (uint64_t i = (uint64_t)lane; i < n; i += 32) out[op + i] = in[ip + i];
    ip += n; op += n;
  };
  auto copy_match = [&](uint64_t off, uint64_t n) {
    if (off == 0 || off > op || op + n > out_len) { bad = true; return; }
    __syncwarp();                                  // the bytes before op are complete
    const uint8_t* from = out + (op - off);
    for (uint64_t i = (uint64_t)lane; i < n; i += 32) out[op + i] = from[i % off];
    op += n;
    __syncwarp();
  };
  if (D.codec == PB_CODEC_SNAPPY) {
    // preamble: decoded length as a varint, then literal / copy elements (tag in the low two bits)
    uint64_t want = 0; int sh = 0;
    for (;;) {
      if (ip >= in_len || sh > 28) { bad = true; break; }
      const uint32_t b = in[ip++];
      want |= (uint64_t)(b & 127u) << sh; sh += 7;
      if (!(b & 128u)) break;
    }
    if (want != out_len) bad = true;
    while (!bad && ip < in_len) {
      const uint32_t tag = in[ip++];
      if ((tag & 3u) == 0) {
        uint64_t n = tag >> 2;
        if (n >= 60) {
          const int nb = (int)n - 59;
          if (ip + nb > in_len) { bad = true; break; }
          n = 0;
          for (int k = 0; k < nb; k++) n |= (uint64_t)in[ip + k] << (8 * k);
          ip += nb;
        }
        copy_literals(n + 1);
      } else if ((tag & 3u) == 1) {
        if (ip + 1 > in_len) { bad = true; break; }
        const uint64_t off = ((uint64_t)(tag >> 5) << 8) | in[ip]; ip += 1;
        copy_match(off, 4 + ((tag >> 2) & 7u));
      } else {
        const int nb = (tag & 3u) == 2 ? 2 : 4;
        if (ip + nb > in_len) { bad = true; break; }
        uint64_t off = 0;
        for (int k = 0; k < nb; k++) off |= (uint64_t)in[ip + k] << (8 * k);
        ip += nb;
        copy_match(off, (tag >> 2) + 1);
      }
    }
  } else {
    if (D.codec == PB_CODEC_LZ4_LENGTH_PREFIXED) {   // lz4-java LZ4CompressorWithLength: decoded length, little-endian int
      if (in_len < 4) bad = true;
      else {
        const uint64_t want = (uint64_t)in[0] | ((uint64_t)in[1] << 8) | ((uint64_t)in[2] << 16) | ((uint64_t)in[3] << 24);
        if (want != out_len) bad = true;
        ip = 4;
      }
    }
    // LZ4 block: token (literal length : match length - 4), [length bytes], literals, offset LE16, [length bytes]; the
    // last sequence ends after its literals
    while (!bad && ip < in_len) {
      const uint32_t token = in[ip++];
      uint64_t lit = token >> 4;
      if (lit == 15) for (;;) { if (ip >= in_len) { bad = true; break; } const uint32_t b = in[ip++]; lit += b; if (b != 255) break; }
      if (bad) break;
      copy_literals(lit);
      if (bad || ip >= in_len) break;
      if (ip + 2 > in_len) { bad = true; break; }
      const uint64_t off = (uint64_t)in[ip] | ((uint64_t)in[ip + 1] << 8); ip += 2;
      uint64_t ml = token & 15u;
      if (ml == 15) for (;;) { if (ip >= in_len) { bad = true; break; } const uint32_t b = in[ip++]; ml += b; if (b != 255) break; }
      if (bad) break;
      copy_match(off, ml + 4);
    }
  }
  if ((bad || op != out_len) && lane == 0) atomicAdd(D.err, 1u);
}

// sorted forward index (docId range pairs) -> big-endian bit-packed dictId stream, so a sorted column can
// be read like any other dictionary column (SortedIndexReaderImpl doubles as the forward index:
// SEGL/segment/index/readers/sorted/SortedIndexReaderImpl.java:37-116).  One thread per output word.
static __global__ void pb_sorted_to_packed_kernel(const int32_t* __restrict__ pairs_le, int32_t card, uint32_t num_docs, int bits,
                                           uint32_t* __restrict__ out_words, uint64_t n_words) {
  for (uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < n_words; w += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t bit0 = w * 32;
    uint64_t first = bit0 / bits;                       // first value overlapping this word
    uint32_t acc = 0;
    for (uint64_t v = first; v * bits < bit0 + 32 && v < num_docs; v++) {
      // dictId of doc v: binary search on end docIds
      int lo = 0, hi = card - 1;
      while (lo < hi) { int mid = (lo + hi) >> 1; if ((uint32_t)pairs_le[2 * mid + 1] < (uint32_t)v) lo = mid + 1; else hi = mid; }
      uint64_t id = (uint64_t)lo;
      long long sh = (long long)(bit0 + 32) - (long long)(v * bits + bits);   // left shift to place value's LSB
      if (sh >= 0) acc |= (uint32_t)(id << sh); else acc |= (uint32_t)(id >> (-sh));
    }
    out_words[w] = pb_bswap32(acc);
  }
}
