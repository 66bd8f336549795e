// Host-callable launchers of every CUDA kernel in libb200exec (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "program.h"

namespace b200 {

// ---- fused pipeline (pipeline.cu) ---------------------------------------------------------------
cudaError_t launch_pipeline(const Program& P, int reg_groups, int grid, int block, size_t smem, cudaStream_t st);
// fused scan->filter->project->aggregate kernel (fused.cuh); *is_static: 1 when an ahead-of-time shape ran
cudaError_t launch_fused_pipeline(const Program& P, const FusedSpec& F, FusedShape shape, int reg_groups, int grid, int block, size_t smem, cudaStream_t st,
                                  int* is_static);
bool fused_rows_ok(const Program& P, int grid, int block, int rows_per_thread);
bool pipeline_add_only(const Program& P, int grid, int block);

// ---- aggregate table (kernels.cu) ----------------------------------------------------------------
struct AccKinds {
  uint8_t kind[VM_MAX_ACC];
  int n;
};
void launch_agg_table_init(const AggTable& T, const AccKinds& kinds, cudaStream_t st);

enum AggOutKind : uint8_t {
  AO_KEY = 0,      // a: key index
  AO_ACC_I128,     // a: acc index, b: count-acc index (valid iff count > 0) or 255
  AO_ACC_I64,      // low 64 bits of an I128 accumulator (SUM(Int64) wraps) ; b as above
  AO_ACC_F64,      // f64 sum ; b as above
  AO_COUNT,        // a: acc index -> Int64/UInt64
  AO_MINMAX_F64,   // order-key -> double ; b count
  AO_AVG_DEC,      // a: sum acc, b: count acc, imm: 10^k multiplier exponent
  AO_AVG_F64,      // a: sum acc (f64), b: count acc
  AO_KEY_PACKED    // a: key index holding a packed short string (OP_STR_PACK8); imm: bit position of the length; aux: 8 B/row chars
};
struct AggOut {
  void* data;
  uint8_t* valid;
  void* aux;
  uint8_t kind;
  uint8_t a, b;
  uint8_t phys;   // output encoding
  int32_t imm;
};
struct AggExtractArgs {
  AggOut out[VM_MAX_OUT];
  int n_out;
  int n_keys;
  unsigned long long* counter;   // device: rows emitted
  unsigned long long cap;        // rows the outputs hold: groups past them are counted, not written
  unsigned int* error;           // device: RunStatus.error
};
void launch_agg_extract(const AggTable& T, const AggExtractArgs& A, cudaStream_t st);

// ---- scans, histograms, scatter/gather ------------------------------------------------------------
// exclusive prefix sum of n uint32 -> uint64 (out[n] = total if out has n+1 slots)
void launch_scan_u32_to_u64(const uint32_t* in, uint64_t* out, int64_t n, uint64_t* scratch /* >= n/1024+2 */, cudaStream_t st);
void launch_histogram_u32(const uint32_t* ids, int64_t n, uint32_t n_bins, unsigned long long* counts, cudaStream_t st);
// dest[i] = cursor[ids[i]]++  (cursor pre-seeded with the exclusive scan of counts)
// stable placement of rows into hash partitions: dest[i] = rows of lower partitions + earlier rows of the same
// partition (input order kept inside a partition, like the reference's BatchPartitioner).  Scratch as for
// radix_sort_pairs_u64; returns the number of launches.
uint64_t launch_partition_dest_stable(const uint32_t* ids, int64_t n, uint32_t n_bins, uint32_t* dest, uint64_t* keys_a, uint32_t* vals_a, uint64_t* keys_b,
                                      uint32_t* vals_b, uint32_t* hist_scratch, uint64_t* scan_scratch, cudaStream_t st);
void launch_scatter_fixed(const void* in, void* out, const uint32_t* dest, int64_t n, int width, cudaStream_t st);
// out[i] = idx[i] >= 0 ? in[idx[i]] : 0 ; valid_out (optional) = idx>=0 && valid_in
void launch_gather_fixed(const void* in, const uint8_t* valid_in, void* out, uint8_t* valid_out, const int64_t* idx, int64_t n, int width, cudaStream_t st);
// the same for up to GATHER_MAX_COLS columns in one launch
static const int GATHER_MAX_COLS = 32;
struct GatherCol {
  const void* in;
  const uint8_t* valid_in;
  void* out;
  uint8_t* valid_out;
  int width;
  int _pad;
  // partition scatter only: when set, row `dst` of partition p is written to (byte address) part_base[p] + dst * width
  // instead of out + dst * width -- the bases may point into ANOTHER GPU's memory (fused shuffle: the scatter kernel
  // stores straight into the owning executor's window over NVLink)
  const unsigned long long* part_base;
};
struct GatherCols {
  GatherCol c[GATHER_MAX_COLS];
  int n;
};
void launch_gather_multi(const GatherCols& cols, const int64_t* idx, int64_t n, cudaStream_t st);
// ingest: int32 / int64 (width 4 / 8) -> sign-extended 16-byte Decimal128 values
void launch_widen_to_i128(const void* in, int width, void* out, int64_t n, cudaStream_t st);
// out[i] = in[i] - in[0] for i < n_plus_1; first_last[0..1] = in[0], in[n_plus_1 - 1] (device memory)
void launch_rebase_offsets(const int32_t* in, int64_t n_plus_1, int32_t* out, int32_t* first_last, cudaStream_t st);
void launch_iota_i64(int64_t* out, int64_t n, cudaStream_t st);

// ---- strings / validity ------------------------------------------------------------------------
void launch_utf8_to_views(const int32_t* offsets, const uint8_t* chars, unsigned long long* views, int64_t n, cudaStream_t st);
void launch_prepack3(const int32_t* offsets, const uint8_t* chars, int64_t n, uint32_t* out, unsigned int* too_long, cudaStream_t st);
void launch_view_lengths(const unsigned long long* views, const uint8_t* valid, uint32_t* lens, int64_t n, cudaStream_t st);
void launch_views_to_utf8(const unsigned long long* views, const uint8_t* valid, const uint64_t* offs64, int32_t* offsets_out, uint8_t* chars_out, int64_t n, cudaStream_t st);
void launch_bitmap_to_bytes(const uint8_t* bitmap, int64_t bit_offset, uint8_t* bytes, int64_t n, cudaStream_t st);
void launch_bytes_to_bitmap(const uint8_t* bytes, uint8_t* bitmap, int64_t n, unsigned long long* null_count, cudaStream_t st);

// ---- hash join --------------------------------------------------------------------------------
struct KeyCol {
  const void* data;
  const uint8_t* valid;
  uint8_t phys;
  uint8_t width;
};
struct JoinKeys {
  KeyCol build[VM_MAX_KEYS];
  KeyCol probe[VM_MAX_KEYS];
  int n_keys;
  int null_equals_null;
};
// ---- one-pass stable radix partition + exchange / export packing (shuffle.cu) ---------------------
static const int PART_MAX_STR_COLS = 16;
static const uint32_t PART_MAX_FANOUT = 4096;   // per-warp counters of the scatter kernel must fit shared memory
struct PartStrCol {
  const void* data;       // views (16 B/row) or Arrow int32 offsets
  const uint8_t* valid;
  int is_view;
  int _pad;
};
struct PartStrCols {
  PartStrCol c[PART_MAX_STR_COLS];
  int n;
};
// Where a row's partition id comes from: a materialised uint32 column (computed by the child's pipeline kernel), or --
// when the shuffle keys are plain integer-like columns -- the key columns themselves: the partition kernels then apply the
// row hash of csrc/common/hash.hpp (first key sets, later keys combine, NULL skips) and `% P` on the fly, and the
// materialising pass disappears.
struct PidSrc {
  const uint32_t* pid;
  KeyCol keys[VM_MAX_KEYS];
  int n_keys;
  // 0: the shuffle's partition function, hash(keys) % P (what the reference computes).  != 0: the key hash is re-mixed with
  // this salt first -- used when rows are partitioned for a purpose of the engine's own (partition-first aggregation) whose
  // input may already be one shuffle partition: without the salt all of its keys agree on hash % P_shuffle and would pile
  // up in the few buckets b with b % P_shuffle == p
  int salt;
};
uint32_t partition_n_tiles(int64_t n);
// tile_hist: [P][n_tiles] u32 (may be nullptr when only totals are wanted); counts: [P] u64, pre-zeroed;
// str_bytes: [sc.n][P] u64, pre-zeroed; pid.pid == nullptr && pid.n_keys == 0 means "everything goes to partition 0"
cudaError_t launch_partition_hist(const PidSrc& pid, int64_t n, uint32_t P, uint32_t* tile_hist, unsigned long long* counts, const PartStrCols& sc,
                                  unsigned long long* str_bytes, cudaStream_t st);
// offsets: exclusive scan of tile_hist (partition-major); cols: every column to move (validity bytes as their own
// width-1 entries; only in/out/width are used); dest_out (optional): the destination row of every input row
cudaError_t launch_partition_scatter(const PidSrc& pid, int64_t n, uint32_t P, const uint64_t* offsets, const GatherCols& cols, uint32_t* dest_out,
                                     cudaStream_t st);
enum PackKind : int32_t { PK_COPY = 0, PK_STR_VIEWS = 1, PK_STR_UTF8 = 2, PK_BITMAP = 3, PK_UTF8_VIEWS = 4 };
struct PackJob {
  const void* src;        // bytes / views / int32 offsets (already positioned at the slice's first row)
  const uint8_t* valid;   // strings: validity bytes of the slice or nullptr
  const uint8_t* chars;   // PK_STR_UTF8: chars base the offsets are relative to
  void* dst;              // PK_COPY: destination; strings: int32 offsets out (rows + 1, starting at 0)
  void* dst2;             // strings: characters out
  uint64_t bytes;         // PK_COPY: bytes to copy; strings: capacity of the character area
  int64_t rows;           // strings, PK_BITMAP
  int32_t kind;
  int32_t _pad;
};
void launch_pack_jobs(const PackJob* jobs_dev, int n_jobs, cudaStream_t st);

void launch_join_build(const uint64_t* build_hash, const uint8_t* build_ok, int64_t n_build, int32_t* heads, uint64_t n_buckets, int32_t* next, cudaStream_t st);
// pass 1: counts per probe row (+ marks); pass 2: write pairs at offsets
void launch_join_probe_count(const JoinKeys& K, const uint64_t* build_hash, const int32_t* heads, uint64_t n_buckets, const int32_t* next,
                             const uint64_t* probe_hash, const uint8_t* probe_ok, int64_t n_probe, uint32_t* counts, uint8_t* build_mark, cudaStream_t st);
void launch_join_probe_write(const JoinKeys& K, const uint64_t* build_hash, const int32_t* heads, uint64_t n_buckets, const int32_t* next,
                             const uint64_t* probe_hash, const uint8_t* probe_ok, int64_t n_probe, const uint64_t* offsets,
                             int64_t* out_build_idx, int64_t* out_probe_idx, cudaStream_t st);
// ---- FilterExec + column projection without the tile VM (filter.cu) ------------------------------------------
static const int FF_MAX_COLS = 16, FF_MAX_OPS = 48, FF_MAX_IMMS = 40, FF_MAX_OUT = 24;
enum FfOpKind : uint8_t { FF_CMP = 0, FF_AND = 1, FF_OR = 2, FF_NOT = 3, FF_FILTER_REG = 4 };
struct FfCol {
  const void* data;       // values / Arrow offsets / views
  const uint8_t* chars;   // PH_UTF8
  uint8_t phys, width;
  uint8_t _pad[6];
};
struct FfOp {
  uint8_t kind;           // FfOpKind
  uint8_t cmp;            // FF_CMP: 0 EQ 1 NE 2 LT 3 LE 4 GT 5 GE
  uint8_t vt;             // FF_CMP: 0 signed 64-bit, 1 signed 128-bit, 2 string (EQ / NE), 3 unsigned 64-bit
  uint8_t filter;         // 1: the result ANDs into the row's pass flag instead of landing in a register
  uint8_t dst;            // bool register (bit of the per-row register word)
  uint8_t a, b;           // FF_CMP: column or immediate index; logic: bool registers
  uint8_t a_imm, b_imm;   // FF_CMP: operand is an immediate
  uint8_t _pad[3];
};
struct FfImm {
  uint64_t lo, hi;        // integers: two's complement 128-bit; strings: device pointer, length
};
struct FastFilterSpec {
  FfCol cols[FF_MAX_COLS];
  FfOp ops[FF_MAX_OPS];
  FfImm imms[FF_MAX_IMMS];
  int n_cols, n_ops, n_out, _pad;
  uint8_t out_col[FF_MAX_OUT];
  void* out_data[FF_MAX_OUT];
  int64_t n_rows;
  unsigned long long* tile_state;   // one look-back word per 1024-row tile, zeroed
  RunStatus* status;
};
cudaError_t launch_fast_filter(const FastFilterSpec& S, int sm_count, cudaStream_t st);

// ---- high-cardinality group-by over plain columns (groupby.cu) ---------------------------------------
static const int GB_MAX_ACC = 8;
struct GroupBySpec {
  FusedCol cols[FUSED_MAX_COLS];   // data + width of every referenced column (no validity, 4 / 8 / 16 bytes wide)
  int n_cols;
  int n_filters;
  int f_col[FUSED_MAX_FILTERS], f_op[FUSED_MAX_FILTERS];   // op: 0 EQ 1 NE 2 LT 3 LE 4 GT 5 GE
  int64_t f_imm[FUSED_MAX_FILTERS];
  int n_keys;                       // 1 or 2 (two keys: both must lie in [0, 2^32), checked per row)
  int key_col[2];
  int n_prod;                       // decimal products: kind 0 a*(lit-b), 1 a*(lit+b), 2 a*b; a_src 1 = previous product
  int p_kind[2], p_a_src[2], p_a_col[2], p_b_col[2];
  int64_t p_lit[2];
  int n_acc;
  int a_src[GB_MAX_ACC], a_col[GB_MAX_ACC];   // src: 0 column, 1 / 2 product, 3 COUNT
  int64_t n_rows;
  AggTable table;
  RunStatus* status;
  // partition-first mode (pf_K > 0): the rows were radix-partitioned by hash(keys) % pf_K beforehand (shuffle.cu) and bucket
  // b aggregates into its own region [b * pf_slots, (b + 1) * pf_slots) of the table, small enough to stay in L2 while the
  // CTAs of that bucket run.  pf_row_start[b .. b+1] = the bucket's rows, pf_cta_start[b .. b+1] = the CTAs that process them
  // (launch_groupby_plan fills both from the partition counts on the device: no host round trip).
  int pf_K;
  unsigned long long pf_slots;                 // power of two
  const unsigned int* pf_cta_start;            // [pf_K + 1]
  const unsigned long long* pf_row_start;      // [pf_K + 1]
};
cudaError_t launch_groupby(const GroupBySpec& S, int sm_count, cudaStream_t st);
// counts[K] -> row_start[K + 1], cta_start[K + 1] (one CTA per GROUPBY_ROWS_PER_CTA rows of a bucket)
static const int GROUPBY_ROWS_PER_CTA = 1024;
cudaError_t launch_groupby_plan(const unsigned long long* counts, int K, unsigned long long* row_start, unsigned int* cta_start, cudaStream_t st);

// ---- single-pass join (join.cu) -----------------------------------------------------------------
struct JoinNode {   // one per build row
  uint64_t tag;     // exact mode: 64-bit image of the (single, integer-like) key; else the row hash
  int32_t next;     // previous head of the bucket, -1 = end of chain
  uint32_t _pad;
};
// exact == true: one integer-like key column, tag = key (build_hash / probe_hash unused)
void launch_join_build2(const JoinKeys& K, bool exact, const uint64_t* build_hash, int64_t n_build, int32_t* heads /* pre-set to -1 */, uint64_t n_buckets,
                        JoinNode* nodes, cudaStream_t st);
// mode bit 0: emit (build row, probe row) pairs -- *counter (pre-zeroed) ends up with the total number of pairs, of
// which the first `cap` were written; bit 1: probe_mark[j] = 1 for probe rows with a match; bit 2: build_mark[i] = 1
void launch_join_probe2(const JoinKeys& K, bool exact, int mode, const JoinNode* nodes, const int32_t* heads, uint64_t n_buckets, const uint64_t* probe_hash,
                        int64_t n_probe, unsigned long long* counter, uint64_t cap, int64_t* out_build_idx, int64_t* out_probe_idx, uint8_t* probe_mark,
                        uint8_t* build_mark, cudaStream_t st);
// compaction helpers: indices of rows whose flag byte == want
void launch_flag_to_u32(const uint8_t* flags, uint8_t want, uint32_t* out, int64_t n, cudaStream_t st);
void launch_select_indices(const uint32_t* flag01, const uint64_t* offs, int64_t* out_idx, int64_t n, cudaStream_t st);
void launch_counts_to_flag(const uint32_t* counts, uint8_t* flags, int64_t n, cudaStream_t st);
void launch_mark_from_idx(const int64_t* idx, int64_t n, uint8_t* marks, cudaStream_t st);

// ---- sort -------------------------------------------------------------------------------------
struct SortWordArgs {
  const void* data;
  const uint8_t* valid;
  uint8_t phys;
  uint8_t asc;
  uint8_t nulls_first;
  int32_t word;   // which 64-bit word of the normalised key (strings / i128 have several); -1 = null rank word
};
void launch_sort_word(const SortWordArgs& A, const uint32_t* perm, uint64_t* out, int64_t n, cudaStream_t st);
// Small inputs (n <= SMALL_SORT_MAX_ROWS): stable sort permutation by direct comparison of up to SMALL_SORT_MAX_KEYS keys
// in ONE launch (rank = number of rows that order before), same ordering as the key-word radix sort: NULL placement
// per key, ascending/descending, IEEE total order for floats, bytewise strings with the shorter prefix first.
static const int SMALL_SORT_MAX_ROWS = 1024;
static const int SMALL_SORT_MAX_KEYS = 8;
struct SmallSortKeys {
  SortWordArgs k[SMALL_SORT_MAX_KEYS];  // `word` unused
  int n_keys;
};
void launch_small_sort(const SmallSortKeys& K, int64_t* perm_out, int64_t n, cudaStream_t st);
void launch_max_view_len(const unsigned long long* views, const uint8_t* valid, int64_t n, unsigned int* out_max, cudaStream_t st);
// stable LSD radix sort of (key, val) pairs on 64-bit keys; ping-pong buffers; returns via *result_in_a
void radix_sort_pairs_u64(uint64_t* keys_a, uint32_t* vals_a, uint64_t* keys_b, uint32_t* vals_b, int64_t n, uint32_t* hist_scratch,
                          uint64_t* scan_scratch, cudaStream_t st, bool* result_in_a, uint64_t* launches);
void launch_iota_u32(uint32_t* out, int64_t n, cudaStream_t st);
void launch_u32_to_i64(const uint32_t* in, int64_t* out, int64_t n, cudaStream_t st);

// ---- Parquet page decode (parquet.cu) ----------------------------------------------------------------
enum PqOutKind : int32_t { PQ_OUT_I32 = 0, PQ_OUT_I64 = 1, PQ_OUT_F64 = 2, PQ_OUT_DEC128 = 3, PQ_OUT_STRVIEW = 4, PQ_OUT_BOOL8 = 5 };
struct PqPage {
  const uint8_t* data;      // page payload in HBM (after the Thrift page header)
  uint32_t n_values;        // values including NULLs (dictionary pages: entries)
  uint32_t def_off, def_len;  // definition-level section inside the payload; len 0 = required column / no levels
  uint32_t val_off, val_len;  // values section
  uint32_t encoding;        // 0 PLAIN, 1 dictionary indices, 2 RLE (BOOLEAN values)
  uint32_t v1_levels;       // 1: data page V1 of a nullable column -- the payload starts with [u32 length][definition levels], values follow
                            //    (the length sits inside the possibly compressed payload, so it is read on the device); val_len = payload bytes
  int64_t row0;             // first row of the page inside the column (dictionary pages: first entry in the dictionary array)
  int64_t dict_base;        // data pages: first entry of their chunk's dictionary
};
struct PqColumn {
  int32_t phys;             // parquet physical type (pq::PhysType)
  int32_t type_length;      // FIXED_LEN_BYTE_ARRAY
  int32_t out_kind;         // PqOutKind
  int32_t _pad;
  void* dict;               // decoded dictionary entries (output type; byte arrays as 16-byte views)
};
struct PqDecompJob {
  const uint8_t* src;   // compressed (or stored) bytes in HBM
  uint8_t* dst;         // where the page payload is rebuilt
  uint32_t src_len, dst_len;
  uint32_t raw_copy;    // 1: plain copy (sections that are never compressed)
  uint32_t _pad;
};
void launch_pq_snappy(const PqDecompJob* jobs, int n_jobs, unsigned int* error, cudaStream_t st);
void launch_pq_levels(const PqPage* pages, int n_pages, uint8_t* valid, uint32_t* nonnull, unsigned long long* total_nonnull, cudaStream_t st);
void launch_pq_page_scan(const uint32_t* nonnull, int n_pages, unsigned long long* dense_base, cudaStream_t st);
void launch_pq_dict(const PqColumn& C, const PqPage* dict_pages, int n_dicts, cudaStream_t st);
void launch_pq_values(const PqColumn& C, const PqPage* pages, int n_pages, const unsigned long long* dense_base, const uint32_t* nonnull, void* out, cudaStream_t st);
void launch_pq_expand(const PqPage* pages, int n_pages, const unsigned long long* dense_base, const uint8_t* valid, const void* dense, void* out, int width,
                      cudaStream_t st);

// ---- synthetic TPC-H input ----------------------------------------------------------------------
void launch_tpch_fixed(int table, int col, int kind, int64_t msf, int64_t row0, int64_t n, void* out, cudaStream_t st);
void launch_tpch_str_len(int table, int col, int64_t msf, int64_t row0, int64_t n, uint32_t* lens, cudaStream_t st);
void launch_tpch_str_fill(int table, int col, int64_t msf, int64_t row0, int64_t n, const uint64_t* offs64, int32_t* offsets, uint8_t* chars, cudaStream_t st);

}  // namespace b200
