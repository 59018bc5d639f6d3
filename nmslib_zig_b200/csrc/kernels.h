// kernels.h -- host-callable launchers of the nmslib_b200 CUDA kernels.
#pragma once
#include <vector>
#include <cuda_runtime.h>
#include <stdint.h>

namespace nb200 {

// ---- options --------------------------------------------------------------------------
// Documented variant selectors, set per process through nmslib_b200_set_option (every variant returns the same
// answers; the tests use them for A/B comparisons):
//   "tc_pair"     1 (default) long rows on CTA pairs / 0 the single-CTA long-row kernel
//   "hnsw_team"   -1 (default) auto / 0 one warp per query / 2, 4 teams of that many warps
//   "force_exact" 0 (default) / 1 CUDA-core exact scan only (read when an index is created)
//   "tc_split"    1 (default) / 0 never switch to split (3xTF32) operands
//   "u8_imma"     1 (default) uint8 rows on the integer tensor pipe / 0 rows widened to TF32 operands
int nb200_option(const char* name, int dflt);
void nb200_set_option(const char* name, int value);
// Timing / debugging knobs (NB200_* environment variables) exist only in -DNB200_EXPERIMENTS builds (the tools);
// the release library never reads them: nb200_env() is then a constant nullptr and the kernels' debug branches
// are compiled out.
#ifdef NB200_EXPERIMENTS
const char* nb200_env(const char* name);
#define NB200_DBG(flags, bit) ((flags) & (bit))
#else
inline const char* nb200_env(const char*) { return nullptr; }
#define NB200_DBG(flags, bit) (false)
#endif

// accumulate/epilogue flavours of the exact scan kernel
enum ScanMode : int { SCAN_L2 = 0, SCAN_NEGDOT = 1, SCAN_COSINE = 2, SCAN_SIFT = 3, SCAN_L1 = 4, SCAN_LINF = 5,
                      SCAN_ANGULAR = 6 };  // L1 / LINF: exact CUDA-core scan only; ANGULAR: cosine ranking, acos at the end

// ---- scan_exact.cu -------------------------------------------------------------------
// db: [n_pad][row_words] words (float32 or packed uint8), rows beyond n are zero padding up
// to a multiple of scan_exact_block_points(); queries alike, padded to a multiple of
// scan_exact_block_queries().  row_words must be a multiple of scan_exact_stage_words().
// partial: [nq][n_split][k] keys, each split's list ascending, KEY_MAX padded.
cudaError_t launch_scan_exact(int mode, const void* db, const void* queries, const void* db_aux,
                              const void* q_aux, int n, int nq, int row_words, int k, uint32_t pos_base,
                              uint64_t* partial, int n_split, int tiles_per_split, cudaStream_t stream,
                              const int* d_nq = nullptr,   // d_nq: query count read on the device (<= nq)
                              uint64_t* glists = nullptr);  // k > scan_exact_smem_k(): scratch of scan_exact_glists_bytes()
// Range mode (batched range queries, mode SCAN_L1 / SCAN_LINF): every query's fixed threshold comes from radii[nq];
// cand / cand_cnt / cut are the candidate lists range_verify_kernel reads (see launch_range_verify), n_split lists
// of list_cap keys per query, written for every query row of the grid (queries padded to 256-query blocks).
cudaError_t launch_scan_exact_range(int mode, const void* db, const void* queries, int n, int nq, int row_words,
                                    uint32_t pos_base, const float* radii, int list_cap, uint64_t* cand, int* cand_cnt,
                                    uint32_t* cut, int n_split, int tiles_per_split, cudaStream_t stream);
int scan_exact_max_k();
int scan_exact_smem_k();
size_t scan_exact_glists_bytes(int nq, int k, int n_split);
int scan_exact_block_queries();
int scan_exact_block_points();
int scan_exact_stage_words();
cudaError_t launch_row_aux(bool is_u8, const void* rows, int n, int row_words, void* out, cudaStream_t stream,
                           const int* d_n = nullptr);

// ---- topk_merge.cu -------------------------------------------------------------------
// Merge `lists` ascending key lists per query into the k best and finalise them.
// key(l, q, e) = keys[l * list_stride + q * query_stride + e]; ids_in (same layout) is
// optional -- when NULL the id is ext_ids[pos - pos_base] (ext_ids NULL: id = pos).
// Outputs are [nq][k]; out_keys / out_counts may be NULL.
cudaError_t launch_merge_topk(const uint64_t* keys, const int32_t* ids_in, int lists, size_t list_stride,
                              size_t query_stride, int nq, int k, int finalize, const int32_t* ext_ids,
                              uint32_t pos_base, uint64_t* out_keys, int32_t* out_ids, float* out_dists,
                              int32_t* out_counts, cudaStream_t stream, const int* d_nq = nullptr);
int merge_topk_max_items();

// gather rows idx[i] of a [*, row_words] array into dst[i] / scatter k-key rows back
// uint8 rows [rows][dim] -> fp32 rows [rows][row_words] (padding columns are left untouched)
cudaError_t launch_widen_u8(const uint8_t* src, size_t rows, int dim, int row_words, float* dst, cudaStream_t stream);
// d_count (optional): row count read on the device (<= count); rows up to the next multiple of `pad` are zero-filled
cudaError_t launch_gather_rows(const uint32_t* src, const int* idx, int count, int row_words, uint32_t* dst,
                               cudaStream_t stream, const int* d_count = nullptr, int pad = 1);
// f2i: the source keys carry f32_ordered(exact-integer float distance), the destination wants i32_ordered (uint8 indexes)
cudaError_t launch_scatter_keys(const uint64_t* src, const int* idx, int count, int k, uint64_t* dst,
                                cudaStream_t stream, const int* d_count = nullptr, int f2i = 0);

// ---- scan_tc.cu (tcgen05 TF32 candidates + exact fp32 re-rank) -------------------------
int tc_block_queries();   // queries per CTA (256): query buffers are padded to this
int tc_block_points();    // database rows per tile (128)
int tc_kblock_words();    // row padding granularity in 32-bit words (32 = 128 bytes)
int tc_max_k();
void tc_candidate_shape(int k, int* kprime, int* cap);
// mode: SCAN_L2 / SCAN_COSINE / SCAN_NEGDOT.  bias[n_pad]; norm2[n] (may be NULL); db_unit: normalised
// copy (cosine only); max_norm_bits: float bits of max |operand row|; inexact_flag: set if not TF32-exact
// nblock: [n_pad][32] |x|^2 as three TF32 pieces (l2 only, else NULL); ones: [128][32] constant A tile for it
cudaError_t launch_tc_prep_db(const float* db, int n, int n_pad, int row_words, int mode, float* bias, float* norm2,
                              float* db_unit, float* nblock, float* ones, unsigned* max_norm_bits,
                              int* inexact_flag, cudaStream_t stream);
// balanced (query block x tile) decomposition: CTAs, work items per CTA, candidate pieces per query block
// bn = database rows per tile of the kernel that will run (tc_block_points() or tc_ts_block_points())
// (the single-CTA long-row kernel, kept behind NB200_TC_PAIR=0 for A/B runs)
void tc_plan(int nq, int n, int k, int sm_count, int bn, int* n_cta, int* work_per_cta, int* s_max, int* aligned);
// long rows on CTA pairs (cta_group::2 MMAs, M256 x N256): plan with tc_ts_plan(nq, n, k, sm_count / 2, &table,
// &n_pairs, &slots, tc_pair_block_points(), 2), upload the table and pass s_max = 2 * slots
bool tc_pair_enabled();   // NB200_TC_PAIR=0 switches back to the single-CTA kernel (A/B runs)
int tc_pair_block_points();
cudaError_t launch_tc_scan_pair(const float* qa, size_t q_pad, const float* dbB, size_t n_pad, const float* nblock,
                                const float* ones, int n, int nq, int row_words, int k, uint32_t pos_base, int n_pairs,
                                const int* d_pieces, int s_max, int kprime, uint64_t* cand, int* cand_cnt,
                                float* cand_thr, uint32_t* gthr, cudaStream_t stream,
                                uint32_t* range_cut = nullptr);  // range mode (see launch_tc_scan_ts)
// rows of at most 128 floats: the prepared queries live in tensor memory (tc_scan_ts_kernel); q = the ORIGINAL
// queries [q_pad][row_words], scaled on the fly; sets *inexact_flag when a valid query row is not TF32-exact
bool tc_ts_supported(int row_words);
int tc_ts_block_points();
// table: n_cta * 8 pieces of {query block, first tile, end tile, candidate slot} (query block -1 ends a CTA's list)
// bn: rows per tile (0 = the TS kernel's); lists_per_piece: candidate lists a piece fills (2 for the pair kernel)
// block_slots: pieces of every query block (its re-rank reads that many x lists_per_piece lists)
void tc_ts_plan(int nq, int n, int k, int sm_count, std::vector<int>* table, int* n_cta, int* s_max, int bn = 0,
                int lists_per_piece = 1, std::vector<int>* block_slots = nullptr);
// kprime: survivors of a compaction (k + margin; the certificate needs the margin); gthr: [q_pad] uint32, filled
// with 0xFF by the caller before every launch (best threshold published per query, shared by all CTAs)
cudaError_t launch_tc_scan_ts(const float* q, const float* dbB, size_t n_pad, const float* nblock, const float* ones,
                              int n, int nq, int row_words, int k, int kprime, float scale, uint32_t pos_base,
                              int n_cta, int s_max, const int* d_pieces, uint64_t* cand, int* cand_cnt,
                              float* cand_thr, uint32_t* gthr, int* inexact_flag, cudaStream_t stream,
                              uint32_t* range_cut = nullptr);
// Range mode of the two scans above (range_cut != NULL): gthr holds every query's fixed threshold T_q
// (launch_tc_range_threshold), lists hold tc_range_cap() keys in position order, and range_cut
// ([q_blocks][s_max][256], written for every list in use instead of cand_thr) receives the position of the first
// survivor a full list dropped (0xFFFFFFFF = none).  k only shapes the plan.
int tc_range_cap();
// mode: SCAN_L2 (take_sqrt: l2, else l2sqr) / SCAN_COSINE / SCAN_ANGULAR / SCAN_NEGDOT; radii: [nq] float radii;
// q: staged queries [q_pad][row_words]; x_max / db_inexact: as for the re-rank's certificate
cudaError_t launch_tc_range_threshold(const float* q, int nq, int row_words, int mode, int take_sqrt, const float* radii,
                                      float x_max, int db_inexact, uint32_t* gthr, cudaStream_t stream);
cudaError_t launch_tc_prep_queries(const float* q, float* out, size_t words, float scale, int* inexact_flag,
                                   cudaStream_t stream);
// qa: prepared queries [q_pad][row_words]; dbB: B operand rows [n_pad][row_words];
// cand: [q_blocks][s_max][256][cap] keys, cand_cnt (zeroed by the caller) / cand_thr: [q_blocks][s_max][256]
cudaError_t launch_tc_scan(const float* qa, size_t q_pad, const float* dbB, size_t n_pad, const float* nblock,
                           const float* ones, int n, int nq, int row_words, int k, uint32_t pos_base, int n_cta,
                           int work_per_cta, int s_max, int aligned, int kprime, uint64_t* cand, int* cand_cnt,
                           float* cand_thr, uint32_t* gthr, cudaStream_t stream);
int tc_rerank_pow2(int n_lists, int cap, int k, int n);  // sort-buffer size of a re-rank launch (a power of two)
cudaError_t launch_tc_rerank(const float* db, const float* queries, const float* db_norm2, int n, int nq,
                             int row_words, int k, int n_split, int mode, uint32_t pos_base, const uint64_t* cand,
                             const int* cand_cnt, const float* cand_thr, float x_max, const int* inexact_flags,
                             uint64_t* out_keys, int* out_cert, cudaStream_t stream,  // mode may be SCAN_ANGULAR
                             int q_begin = 0, int q_count = -1, int n_lists = -1,  // a query range whose blocks use
                             float eps_override = 0.f,  // only the first n_lists lists; eps: error band of split operands
                             int* fb_count = nullptr, int* fb_idx = nullptr,  // device-side list of uncertified queries
                             const uint8_t* db_u8 = nullptr, const uint8_t* q_u8 = nullptr,  // byte rows (uint8 on the integer pipe)
                             float abs_err = 0.f, int int_keys = 0);  // absolute pass-1 error bound; int-ordered out keys
// ---- uint8 rows on the integer tensor pipe (tcgen05.mma.kind::i8; scan_tc.cu: tc_scan_u8_kernel) ----
// q / db: byte rows of 128; digits: [n_pad][32] norm digits (launch_u8_norm_digits) of V(x) = m_half - ceil(|x|^2 / 2);
// candidates / thresholds / gthr as for launch_tc_scan_ts (ranks = |x|^2 - 2 q.x + (|x|^2 odd), exact even integers)
int u8_imma_max_norm2();  // largest max |x|^2 the digit block can carry
cudaError_t launch_u8_max_norm(const int* norm2, int n, int* d_out, cudaStream_t stream);
cudaError_t launch_u8_norm_digits(const int* norm2, int n, int n_pad, int m_half, uint8_t* out, cudaStream_t stream);
cudaError_t launch_tc_scan_u8(const uint8_t* q, const uint8_t* db, const uint8_t* digits, size_t n_pad, int n, int nq, int k,
                              int kprime, int m_half, uint32_t pos_base, int n_cta, int s_max, const int* d_pieces,
                              uint64_t* cand, int* cand_cnt, float* cand_thr, uint32_t* gthr, cudaStream_t stream,
                              uint32_t* range_cut = nullptr);  // range mode (see launch_tc_scan_ts)
// range mode of launch_tc_scan_u8: gthr[i] = the int bits of query i's accumulator threshold (a row passes when
// acc > T_acc) for the floored radius radii[i]; q: staged byte queries [q_pad][128]
cudaError_t launch_tc_range_threshold_u8(const uint8_t* q, int nq, const float* radii, int m_half, uint32_t* gthr,
                                         cudaStream_t stream);
// 3xTF32 operand split: dst[r] = [hi | lo | hi] (layout 0, database) or [hi | hi | lo] (layout 1, queries) of
// scale * src[r], hi = the TF32-exact part, lo = the TF32-exact part of the rest; dst rows are 3 * row_words long
cudaError_t launch_tc_split_rows(const float* src, size_t rows, int row_words, float scale, int layout, float* dst,
                                 cudaStream_t stream);

// ---- range_scan.cu (one query, every row within the radius, in position order) ----------
// dist_tmp: [n] scratch; out_ids / out_dists: [capacity] device buffers; *out_count <= capacity
cudaError_t launch_range_scan(const float* db, const float* query, const float* db_norm2, const int32_t* ext_ids, int n,
                              int row_words, int mode, int take_sqrt, float radius, int capacity, float* dist_tmp,
                              int32_t* out_ids, float* out_dists, int* out_count, cudaStream_t stream);
// Batched range queries, verification of the tensor-core candidates (one block per query of [q0, q0 + count)):
// cand / cand_cnt / cut: the range-mode lists of launch_tc_scan_ts / _pair (s_max lists per 256-query block of
// list_cap keys); only candidates below the smallest cut are evaluated, with the distance code of launch_range_scan.
// Outputs in CSR form: query q writes at most caps[q] hits at out_off[q] and *out_count[q]; a query that cannot be
// certified (a list overflowed and fewer than caps[q] hits lie below the cut) is appended to fb_idx / *fb_count.
cudaError_t launch_range_verify(const float* db, const float* queries, const int32_t* ext_ids, int row_words, int mode,
                                int take_sqrt, uint32_t pos_base, const float* radii, const int* caps,
                                const int64_t* out_off, const uint64_t* cand, const int* cand_cnt, const uint32_t* cut,
                                int s_max, int list_cap, int q0, int count, int32_t* out_ids, float* out_dists,
                                int* out_count, int* fb_count, int* fb_idx, cudaStream_t stream);

// ---- hnsw_search.cu ------------------------------------------------------------------
struct HnswDeviceGraph {
  const void* vectors;       // [n][row_words] words: float32 (cosine: unit-norm rows, as the reference stores them)
                             // or, dist_kind 3, packed uint8 rows
  const int32_t* links0;     // [n][maxM0]
  const int32_t* links0_cnt; // [n]
  const int32_t* upper;      // concatenated upper-level lists: per level (maxM+1) ints, count first
  const int64_t* upper_off;  // [n] offset into `upper`, -1 when the node lives on level 0 only
  const int32_t* ext_ids;    // [n]
  int n, dim, row_words, maxM, maxM0, maxlevel, enterpoint;
  int dist_kind;             // 0 squared L2, 1 cosine on unit vectors, 2 negative dot product, 3 squared L2 of uint8 rows
};
// One warp per query.  queries: [nq][row_words] words laid out like the rows.  visited: [slots][n] epoch bytes,
// epochs: [slots] current epoch.  out_keys: [nq][k] (ordered(distance) << 32 | internal position), counters: [2]
// atomics (distance evaluations, expansions), may be NULL.
cudaError_t launch_hnsw_search(const HnswDeviceGraph& g, const void* queries, int nq, int k, int ef,
                               uint8_t* visited, int* slot_epoch, int slots, uint64_t* out_keys,
                               unsigned long long* counters, cudaStream_t stream);
int hnsw_max_ef();
int hnsw_warps_per_block();

}  // namespace nb200
