/*
 * genedex_b200.h -- C ABI of the B200-native batched FM-index search engine.
 *
 * This is the drop-in boundary for genedex's batched search path.  The reference crate has no FFI
 * of its own; the seam is the crate-private call
 *     FmIndex::cursors_for_many_queries -> BatchComputedCursors   (src/lib.rs:241-246)
 * plus FmIndex::locate_interval (src/lib.rs:187-197).  Every entry point below names the reference
 * item it replaces (file:line relative to the genedex source tree).  INTEGRATION.md shows the Rust
 * `extern "C"` block + safe wrapper a maintainer would add to keep the crate's public API.
 *
 * Conventions
 *   - plain pointers and sizes only; all functions return a gdx_status (0 = OK) and never unwind;
 *   - caller owns every input buffer for the duration of the call only;
 *   - outputs whose size is known up front are caller-allocated; variable-size hit arrays are
 *     library-allocated pinned host memory released with gdx_free_hits();
 *   - re-entrant: any number of host threads may call into one gdx_index concurrently
 *     (the reference's search methods take &self and FmIndex is Send + Sync);
 *   - the library requires a CUDA device (sm_100a).  There is no CPU fallback: without a device
 *     every compute entry point returns GDX_ERR_CUDA.
 */
#ifndef GENEDEX_B200_H
#define GENEDEX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GDX_ABI_VERSION 2

typedef enum gdx_status {
    GDX_OK = 0,
    /* the reference panics "symbol in io representation should be valid" (src/alphabet.rs:195-198);
     * gdx_last_error_query() gives the index of the first offending query of the call */
    GDX_ERR_INVALID_SYMBOL = 1,
    GDX_ERR_BAD_ARG = 2,
    GDX_ERR_CUDA = 3,
    GDX_ERR_OOM = 4,
    GDX_ERR_TEXT_TOO_LONG = 5, /* src/construction/mod.rs:34 assert */
    GDX_ERR_UNSUPPORTED = 6,
    GDX_ERR_BUSY = 7           /* an accelerator cannot be rebuilt / freed while queries run on the handle */
} gdx_status;

/* IndexStorage `I` of the reference (src/construction/mod.rs:59-73,146-252). It bounds the total
 * text length exactly like the reference; query results do not depend on it. */
typedef enum gdx_storage { GDX_I32 = 0, GDX_U32 = 1, GDX_I64 = 2 } gdx_storage;

/* where the suffix array is built (construction is not part of the search path) */
typedef enum gdx_construction {
    GDX_CONSTRUCT_HOST = 0,  /* SA-IS on the host (the reference: libsais on the host)          */
    GDX_CONSTRUCT_DEVICE = 1,/* prefix-doubling radix sort on the GPU (n < 2^32 - 1)            */
    GDX_CONSTRUCT_AUTO = 2   /* device when the text and the sort scratch (~36 B/symbol) fit    */
} gdx_construction;

/* src/alphabet.rs:24-28: 256-entry IO->dense table (0 = not in the alphabet; dense 0 is the
 * sentinel), number of dense symbols incl. the sentinel, and how many of them may be searched. */
typedef struct gdx_alphabet {
    uint8_t io_to_dense[256];
    uint32_t num_dense_symbols;
    uint32_t num_searchable_dense_symbols;
} gdx_alphabet;

/* src/config.rs:9-15,72-82 (defaults: sampling rate 4, lookup depth 0, Balanced) */
typedef struct gdx_config {
    uint32_t storage;                /* gdx_storage */
    uint32_t suffix_array_sampling_rate;
    uint32_t lookup_table_depth;
    uint32_t performance_priority;   /* accepted for API parity; never changes a query result */
    uint32_t construction;           /* gdx_construction */
    int32_t device;                  /* CUDA device ordinal, -1 = current device */
    uint32_t flags;                  /* GDX_FLAG_* */
    /* Device memory the optional accelerators of a replica (dense suffix array, seed table; see
     * gdx_index_set_*) may take together, in bytes.  0 = automatic: each accelerator is built when it needs
     * at most a quarter of the device memory that is free at that moment.  The budget is stored in the
     * index image, so replicas, adopted and loaded indexes follow the same policy. */
    uint64_t accelerator_budget_bytes;
} gdx_config;

/* re-check the device-built suffix array in O(n) (permutation + order) before it is used */
#define GDX_FLAG_VERIFY_SUFFIX_ARRAY 1u
/* do not keep the packed text in the device image (saves n/2 bytes for sigma <= 16, n otherwise);
 * count/locate then run every LF step instead of finishing one-row intervals by a text comparison.
 * Results are identical either way. */
#define GDX_FLAG_NO_TEXT 2u
/* do not keep the sampled inverse suffix array (n / rate entries, only kept together with the text):
 * cursors_for_many_queries then runs every LF step. Results are identical either way. */
#define GDX_FLAG_NO_INVERSE_SAMPLES 4u
/* never build the dense suffix array accelerator (see gdx_index_set_dense_suffix_array) for this index */
#define GDX_FLAG_NO_DENSE_SUFFIX_ARRAY 8u
/* never build the seed table accelerator (see gdx_index_set_seed_table_depth) for this index */
#define GDX_FLAG_NO_SEED_TABLE 16u
/* never build the row context table accelerator (see gdx_index_set_row_context_table) for this index */
#define GDX_FLAG_NO_ROW_CONTEXT_TABLE 32u

/* src/lib.rs:331-335 Hit { text_id, position } */
typedef struct gdx_hit {
    uint64_t text_id;
    uint64_t position;
} gdx_hit;
/* the same for texts shorter than 2^32 symbols: half the bytes per hit on the way back from the GPU */
typedef struct gdx_hit32 {
    uint32_t text_id;
    uint32_t position;
} gdx_hit32;

/* How the symbols of a query batch are stored. */
typedef enum gdx_query_encoding {
    /* one IO byte per symbol, translated through the alphabet on the device (the reference's input) */
    GDX_QUERIES_IO_BYTES = 0,
    /* 2 bits per symbol, code = dense symbol - 1, symbol k of the batch at bits [2(k%4), 2(k%4)+2) of byte k/4.
     * Only for alphabets with at most 4 searchable symbols (every DNA alphabet, alphabet.rs:251-300) and only
     * for batches made of searchable symbols (gdx_pack_queries checks that).  With fewer than 4 searchable
     * symbols, a query holding a code >= the number of searchable symbols fails the call with
     * GDX_ERR_INVALID_SYMBOL, wherever in the query the code sits.  A quarter of the PCIe bytes:
     * for callers that keep their reads packed.  IO-byte batches are packed by the library itself while it
     * stages them (see gdx_count_many). */
    GDX_QUERIES_PACKED_2BIT = 1
} gdx_query_encoding;

/* A batch of queries: query i = symbols [offsets[i], offsets[i+1]) of the batch's symbol stream.
 * offsets == NULL means every query has length fixed_len and query i starts at symbol i * fixed_len
 * (+ first_symbol).  With GDX_QUERIES_IO_BYTES symbol k is bytes[k].
 * offsets must not decrease and the symbols [offsets[0], offsets[nq]) must exist; the host entry points do not
 * scan the array (60 M entries would cost more than the search) -- chunk boundaries are checked on the host and
 * every query against its uploaded chunk on the device, so a broken array fails with GDX_ERR_BAD_ARG
 * (gdx_last_error_query names the query) and nothing outside the batch is read.  Device-resident batches
 * (gdx_count_many_device ...) are the caller's contract.
 * Replaces `impl IntoIterator<Item = Q: AsRef<[u8]>>` of src/lib.rs:155-158,179-182,241-244. */
typedef struct gdx_queries {
    const uint8_t *bytes;
    const uint64_t *offsets; /* nq + 1 entries, or NULL */
    uint64_t fixed_len;
    uint64_t nq;
    uint32_t encoding;       /* gdx_query_encoding */
    uint32_t first_symbol;   /* fixed-length batches: stream index of the first symbol of query 0 (sub-batches of a
                              * packed stream need not start on a byte boundary); 0 otherwise */
} gdx_queries;

/* The host-side structures of a constructed reference index, in the reference's own layout
 * (src/lib.rs:93-100): used to move an index built (or loaded from a savefile) by the Rust crate
 * onto the GPU.  Integers of type `I` are passed widened to 64 bit. */
typedef struct gdx_parts {
    gdx_alphabet alphabet;
    uint32_t storage;
    uint64_t text_len;                    /* incl. one sentinel per text, src/lib.rs:292-294       */
    const uint64_t *count;                /* num_dense_symbols + 1 entries, src/lib.rs:95          */
    /* CondensedTextWithRankSupport<I, Block64>, src/text_with_rank_support/condensed.rs:24-30     */
    const uint64_t *interleaved_blocks;   /* ceil((n+1)/64) * ceil(log2 sigma) words               */
    const uint16_t *interleaved_block_offsets; /* ceil((n+1)/64) * sigma (may be NULL: recomputed) */
    /* SampledSuffixArray, src/sampled_suffix_array.rs:18-23                                       */
    const uint64_t *sampled_suffix_array; /* ceil(n / rate) entries, widened; or NULL and ...      */
    uint32_t sampling_rate;
    const uint64_t *text_border_rows;     /* keys of text_border_lookup                            */
    const uint64_t *text_border_positions;/* values of text_border_lookup                          */
    uint64_t num_text_borders;
    /* TexdIdSearchTree, src/text_id_search_tree.rs:6-9                                            */
    const uint64_t *sentinel_indices;
    uint64_t num_texts;
    uint32_t lookup_table_depth;          /* tables are re-derived on the device                   */
    /* ... the crate's own `suffix_array_data: Vec<u32>` (sampled_suffix_array.rs:18-23) as it is for the
     * 32-bit storage types: no widened copy needed.  Exactly one of the two sample pointers is set. */
    const uint32_t *sampled_suffix_array_u32;
    uint32_t flags;                       /* GDX_FLAG_NO_DENSE_SUFFIX_ARRAY | GDX_FLAG_NO_SEED_TABLE | GDX_FLAG_NO_ROW_CONTEXT_TABLE */
    uint64_t accelerator_budget_bytes;    /* as gdx_config.accelerator_budget_bytes                */
    /* Which TextWithRankSupport `interleaved_blocks` comes from (the crate's four type aliases, lib.rs:104-113):
     *   GDX_RANK_CONDENSED: [position group][bit plane] Blocks, NUM_BITS positions per group (condensed.rs:24-47);
     *   GDX_RANK_FLAT:      [position group][dense symbol] one-hot Blocks, NUM_BITS - 16 positions per group, the
     *                       bit of position j at index j + 16 of the Block, low 16 bits = block offset
     *                       (flat.rs:24-52, block.rs:3,122-134).
     * block_bits = Block::NUM_BITS: 64 (Block64) or 512 (Block512 = eight little-endian u64, block.rs:66-134);
     * 0 means 64.  Every variant answers every rank identically (tests/text_with_rank_support.rs:69-75), so all
     * of them become the same device records; block / superblock offsets are recomputed on the device. */
    uint32_t rank_variant;
    uint32_t block_bits;
} gdx_parts;

typedef enum gdx_rank_variant { GDX_RANK_CONDENSED = 0, GDX_RANK_FLAT = 1 } gdx_rank_variant;

typedef struct gdx_index gdx_index;

typedef struct gdx_index_info {
    uint64_t text_len;
    uint64_t num_texts;
    uint32_t num_dense_symbols;
    uint32_t num_searchable_dense_symbols;
    uint32_t storage;
    uint32_t sampling_rate;
    uint32_t lookup_table_depth;
    uint32_t rank_layout;          /* 0: 32 B / 64 positions, 1: generic / 128 positions */
    uint32_t rank_record_bytes;
    uint32_t rank_positions_per_record;
    int32_t device;
    uint64_t image_bytes;          /* size of the device image */
    uint64_t rank_bytes, sample_bytes, lookup_bytes;
    uint64_t num_samples, num_text_borders;
    uint64_t text_bytes;           /* packed text section, 0 if absent */
    uint64_t inverse_sample_bytes; /* sampled inverse suffix array, 0 if absent */
    uint64_t dense_suffix_array_bytes; /* device-only accelerator outside the image, 0 if absent */
    uint64_t seed_table_bytes;         /* device-only accelerator outside the image, 0 if absent */
    uint32_t seed_table_depth;         /* 0 if absent */
    uint32_t row_context_entry_bytes;  /* row context table: bytes per text position (16), 0 if absent */
    uint32_t compact_seed_depth;       /* compact seed level of the seed table (see gdx_index_set_seed_table_depth), 0 if absent */
    uint64_t compact_seed_bytes;       /* device-only accelerator outside the image, 0 if absent */
} gdx_index_info;

/* counters of the last search / locate call on this thread (feeds the roofline arithmetic) */
typedef struct gdx_stats {
    uint64_t queries;
    uint64_t lf_steps;       /* backward-search steps executed (2 rank queries each) */
    uint64_t hits;
    uint64_t walk_steps;     /* LF steps executed by the locate walk                 */
    double kernel_ms_search; /* CUDA-event time of the search kernel(s)              */
    double kernel_ms_locate; /* CUDA-event time of the locate kernels                */
    uint64_t kernel_launches;
    uint64_t verified_queries; /* queries finished by one text comparison instead of LF steps */
    uint64_t locate_walk_steps;/* the part of walk_steps spent in the locate kernel            */
    uint64_t packed_queries;   /* queries that crossed PCIe 2-bit packed (host packer or pre-packed input) */
    uint64_t exception_queries;/* queries of packed chunks re-run from their IO bytes (hold an unencodable byte) */
    uint64_t h2d_bytes;        /* bytes copied host -> device by the call                      */
    uint64_t d2h_bytes;        /* bytes copied device -> host by the call                      */
    uint64_t shards;           /* replicas that worked on the call (1 unless *_sharded)        */
} gdx_stats;

uint32_t gdx_abi_version(void);
const char *gdx_last_error_message(void); /* thread local */
uint64_t gdx_last_error_query(void);      /* thread local */
int32_t gdx_device_count(void);

/* ---- construction: FmIndexConfig::construct_index (src/config.rs:63-69 -> src/lib.rs:118-142) -- */
/* texts: concatenated IO bytes; text_offsets: num_texts + 1 entries. */
gdx_status gdx_index_build(const uint8_t *texts, const uint64_t *text_offsets, uint64_t num_texts,
                           const gdx_alphabet *alphabet, const gdx_config *config, gdx_index **out);

/* Upload an index that the reference crate constructed on the host (src/lib.rs:93-100). */
gdx_status gdx_index_create_from_parts(const gdx_parts *parts, int32_t device, gdx_index **out);

/* Same, from the BWT in dense representation instead of the bit planes (n bytes). */
gdx_status gdx_index_create_from_bwt(const uint8_t *bwt, const gdx_parts *parts, int32_t device,
                                     gdx_index **out);

/* Construction utility: suffix array of a dense text (0 = sentinel, ordinary symbol; end of text
 * sorts first -- the libsais convention the reference relies on, construction/mod.rs:88-103),
 * computed on the host (SA-IS) or on the device (prefix doubling). */
gdx_status gdx_suffix_array(const uint8_t *dense_text, uint64_t n, uint32_t num_dense_symbols,
                            uint32_t where /* gdx_construction */, int32_t device, uint64_t *sa_out);

/* Read back parts of a device index (export / interop utilities, not on the search path):
 * the BWT in dense representation (text_len bytes, host buffer) recovered from the rank records
 * with symbol_at (src/text_with_rank_support/condensed.rs:343-362), and count[] (lib.rs:95). */
gdx_status gdx_index_download_bwt(const gdx_index *idx, uint8_t *bwt_out);
gdx_status gdx_index_get_count(const gdx_index *idx, uint64_t *count_out /* num_dense_symbols + 1 */);
/* the sampled suffix array widened to 64 bit (info.num_samples entries,
 * src/sampled_suffix_array.rs:18-23) and text_border_lookup sorted by row (info.num_text_borders) */
gdx_status gdx_index_download_samples(const gdx_index *idx, uint64_t *samples_out);
gdx_status gdx_index_download_text_borders(const gdx_index *idx, uint64_t *rows_out, uint64_t *positions_out);

/* Construction utility: concatenate + densely encode the texts with one 0 sentinel after each text
 * (src/construction/mod.rs:255-308), sentinel positions and count[] (src/construction/mod.rs:318-336).
 * dense_out: total text length + num_texts bytes; sentinels_out: num_texts; count_out: sigma + 1. */
gdx_status gdx_concat_texts(const uint8_t *texts, const uint64_t *text_offsets, uint64_t num_texts,
                            const gdx_alphabet *alphabet, uint8_t *dense_out, uint64_t *sentinels_out,
                            uint64_t *count_out);

void gdx_index_destroy(gdx_index *idx);
gdx_status gdx_index_get_info(const gdx_index *idx, gdx_index_info *out);

/* Dense suffix array accelerator (memory for speed, B200: 180 GB of HBM).  The index keeps the sampled
 * suffix array the configuration asks for (sampled_suffix_array.rs:10-16) -- that is what is saved,
 * exported and replicated.  On top of it a replica can hold SA[row] for EVERY row (4 B per symbol, 8 B
 * beyond 2^32 - 1 symbols), derived on the device from the samples in a fraction of a second:
 * resolving a row (locate, and the text verification of count/locate) is then one load instead of an
 * LF-walk of up to rate - 1 steps plus a load.  Results are identical with and without it.
 * It is built automatically after construction / load / adopt / replicate when the policy of the index
 * allows it: GDX_FLAG_NO_DENSE_SUFFIX_ARRAY never; gdx_config.accelerator_budget_bytes when set, else at most a
 * quarter of the free device memory.  The policy travels with the image (replicas, files).  The environment
 * variable GDX_DENSE_SA (0 never, 1 always) overrides it for measurements.
 * on != 0 builds it now (GDX_ERR_OOM if it does not fit), on == 0 frees it.  Returns GDX_ERR_BUSY while host-buffer
 * queries run on the handle; the caller must also have drained its own *_device launches. */
gdx_status gdx_index_set_dense_suffix_array(gdx_index *idx, int32_t on);

/* Seed table accelerator (memory for speed).  The index keeps the lookup tables of the configured depth
 * (lookup_table.rs:19-23) -- that is what is saved, exported and replicated, and what decides every
 * error behaviour.  On top of it a replica can hold ONE level of a deeper lookup table (depth d: ns^d
 * entries of 8 B, 16 B beyond 2^32 - 1 symbols), filled on the device level by level with the same
 * rule as the reference (lookup_table.rs:225-258).  A query whose last d symbols are all searchable starts
 * from that entry instead of the configured table + LF steps; the entry is bit for bit the interval those
 * steps produce (also when it is empty), every other query takes the configured path.  Results, error
 * behaviour and reported lookup_table_depth are unchanged.
 * Built automatically after construction / load / adopt / replicate with the largest d such that
 * ns^d <= 4 * text length (at most four entries per text position), under the same policy as the dense suffix array (GDX_FLAG_NO_SEED_TABLE,
 * gdx_config.accelerator_budget_bytes, else a quarter of the free memory; GDX_SEED_TABLE=0 / =d overrides it
 * for measurements).  depth > configured depth (re)builds it at that depth now (GDX_ERR_OOM /
 * GDX_ERR_UNSUPPORTED if it does not fit), any smaller depth just frees it.  GDX_ERR_BUSY as above.
 * The seed table brings a compact seed level: the interval of every d-mer two or more symbols deeper, in about
 * 2 bits per d-mer (groups of 224 d-mers in 64 B, exception records for d-mers of more than two rows).  Count
 * and locate queries whose last d symbols are all searchable start from it; cursors never do.  d is the largest
 * depth with ns^d <= 32 * text length whose level fits the budget when one is set, else half of the free memory.
 * It needs the text section, a text shorter than 2^32 symbols and 32-bit entries, is built last, and is rebuilt
 * and freed together with the seed table (also by GDX_FLAG_NO_SEED_TABLE and GDX_SEED_TABLE=0). */
gdx_status gdx_index_set_seed_table_depth(gdx_index *idx, int32_t depth);

/* Row context table accelerator (memory for speed; alphabets with at most 4 searchable symbols, texts shorter than
 * 2^32 symbols, needs the text section).  One 16-byte entry per suffix array row: SA[row] and the 45 text symbols in
 * front of that position as 2-bit codes (+ how many of them are searchable symbols of the same text).  The text
 * verification of count / locate (below) then decides a one-row interval from ONE random 16-byte read instead of the
 * suffix array entry plus the text window behind it -- two dependent DRAM lines less the one.  Queries longer than 64
 * symbols, queries with more than 45 symbols left to compare, and contexts that run into `N` / a text border fall
 * back to the symbol-by-symbol text comparison, so results and error behaviour are identical with and without it.
 * Derived on the device from the suffix array and the text; not part of the image, of files or of what is replicated.
 * Built automatically last, after the other two accelerators, when it fits what they left: GDX_FLAG_NO_ROW_CONTEXT_TABLE
 * never; gdx_config.accelerator_budget_bytes when set, else at most half of the free device memory (GDX_ROW_CONTEXT =
 * 0 / 1 overrides the policy for measurements).  on != 0 builds it now (GDX_ERR_OOM / GDX_ERR_UNSUPPORTED), on == 0
 * frees it.  GDX_ERR_BUSY as above. */
gdx_status gdx_index_set_row_context_table(gdx_index *idx, int32_t on);

/* Text verification (needs the text section of the image, i.e. no GDX_FLAG_NO_TEXT): count / locate finish an
 * interval that has narrowed to one row by resolving SA[row] and comparing the rest of the query with the
 * text instead of one LF step per remaining symbol.  On by default (GDX_VERIFY=0 changes the default);
 * on == 0 makes every query run every LF step, exactly the reference's sequence of rank queries
 * (batch_computed_cursors.rs:62-70).  Results are identical either way.  GDX_ERR_BUSY as above. */
gdx_status gdx_index_set_text_verification(gdx_index *idx, int32_t on);

/* ---- index files: FmIndex::save_to_file / load_from_file (src/lib.rs:296-327) -------------------------
 * The crate serialises its host structs with the `savefile` crate (schema version 0); that byte format
 * is owned by an un-vendored dependency and no reference test pins it, so this is an own versioned
 * container (magic "GDXFILE1" + image header + device image + caller blob), NOT savefile-compatible.
 * `user_data` is an opaque blob of the host language binding (e.g. the alphabet's dense->io table). */
gdx_status gdx_index_save_to_file(const gdx_index *idx, const char *path, const void *user_data,
                                  uint64_t user_bytes);
gdx_status gdx_index_load_from_file(const char *path, int32_t device, gdx_index **out, void *user_data_out,
                                    uint64_t user_capacity, uint64_t *user_bytes_out);

/* ---- replication (no counterpart in the reference; SURVEY 8e) ----------------------------------
 * The device image is one contiguous allocation described by an opaque POD header.  A replica on
 * another GPU (or in another process) is made by copying header + image bytes, e.g. with one
 * ncclBroadcast from rank 0, and adopting them.  `image` must stay valid while the index lives
 * (own_image = 0) or is freed with cudaFree by gdx_index_destroy (own_image != 0). */
uint64_t gdx_index_header_bytes(void);
gdx_status gdx_index_export(const gdx_index *idx, void *header_out, const void **device_image,
                            uint64_t *image_bytes);
gdx_status gdx_index_adopt_image(const void *header, void *device_image, int32_t device,
                                 int32_t own_image, gdx_index **out);
/* Single process, several GPUs: full replicas of `idx` on `devices` with ONE grouped ncclBroadcast of the
 * device image from the source GPU over NVLink (ncclCommInitAll over the source device + the targets; NCCL is
 * loaded at run time from libnccl.so.2).  A target equal to the source device gets a device-to-device copy.
 * If NCCL cannot be loaded the copies go through cudaMemcpyPeer; gdx_replicate_transport() names what the
 * last call on this thread used ("nccl", "peer").  Every replica then derives its own accelerators
 * (SURVEY 8e: no collective on the query path). */
gdx_status gdx_index_replicate(const gdx_index *idx, const int32_t *devices, int32_t n_devices,
                               gdx_index **out_replicas);
const char *gdx_replicate_transport(void);

/* One process per GPU: rank 0 creates an NCCL unique id (128 bytes), hands it to the other ranks out of band
 * (MPI, torch.distributed, a file, ...), then EVERY rank calls gdx_index_broadcast: the library joins the
 * communicator (ncclCommInitRank), broadcasts image header + device image from rank `root` and adopts them.
 * `src` is the root's index (NULL elsewhere).  *out: a new replica on `device`; on the root it is `src` itself
 * (no copy, do not destroy it twice). */
#define GDX_NCCL_UNIQUE_ID_BYTES 128
gdx_status gdx_nccl_unique_id(void *id_out);
gdx_status gdx_index_broadcast(const gdx_index *src, const void *unique_id, int32_t rank, int32_t world,
                               int32_t root, int32_t device, gdx_index **out);

/* ---- batched search with host buffers ----------------------------------------------------------*/
/* FmIndex::cursors_for_many_queries (src/lib.rs:241-246): intervals [start,end) in input order. */
gdx_status gdx_cursors_many(const gdx_index *idx, const gdx_queries *queries, uint64_t *starts,
                            uint64_t *ends);
/* FmIndex::count_many (src/lib.rs:155-161).
 * Large IO-byte batches over an alphabet with <= 4 searchable symbols are packed to 2 bits per symbol by a
 * pool of host threads while they are staged into pinned memory (GDX_HOST_THREADS, default: the CPUs of the
 * process), so a quarter of the bytes cross PCIe; queries holding any other byte (invalid, or valid but not
 * searchable such as `N`) are re-run from their IO bytes, which keeps the reference's lazy invalid-symbol
 * behaviour exact.  Results of large batches cross PCIe as uint32 when the text is shorter than 2^32. */
gdx_status gdx_count_many(const gdx_index *idx, const gdx_queries *queries, uint64_t *counts);
/* the same with uint32 results written straight into the caller's arrays (GDX_ERR_UNSUPPORTED for texts of
 * 2^32 symbols or more) */
gdx_status gdx_count_many_u32(const gdx_index *idx, const gdx_queries *queries, uint32_t *counts);
gdx_status gdx_cursors_many_u32(const gdx_index *idx, const gdx_queries *queries, uint32_t *starts,
                                uint32_t *ends);
/* Packs an IO-byte batch to GDX_QUERIES_PACKED_2BIT with the library's host packer (for callers that reuse
 * a batch or keep reads packed).  packed_out: gdx_packed_bytes(total symbols) bytes, symbol k of the batch at
 * stream index k (offsets / fixed_len stay valid for the packed batch).  *first_unencodable = index of the
 * first query holding a byte without a 2-bit code, or UINT64_MAX; such a batch must be searched as IO bytes. */
uint64_t gdx_packed_bytes(uint64_t total_symbols);
gdx_status gdx_pack_queries(const gdx_index *idx, const gdx_queries *io_queries, uint8_t *packed_out,
                            uint64_t *first_unencodable);
/* The packer itself, without an index (host only, no GPU needed): n IO bytes -> (n + 3) / 4 packed bytes; the
 * positions of bytes without a 2-bit code (packed as 0) go to exception_positions (up to `capacity`, sorted),
 * their number to *num_exceptions. */
gdx_status gdx_pack_symbols(const gdx_alphabet *alphabet, const uint8_t *io_bytes, uint64_t n,
                            uint8_t *packed_out, uint64_t *exception_positions, uint64_t capacity,
                            uint64_t *num_exceptions);
/* FmIndex::locate_many (src/lib.rs:179-185): CSR result; hit_offsets has nq + 1 entries; the hits
 * of query i are hits[hit_offsets[i] .. hit_offsets[i+1]) in the reference's SA-row order. */
gdx_status gdx_locate_many(const gdx_index *idx, const gdx_queries *queries, uint64_t *hit_offsets,
                           gdx_hit **hits, uint64_t *num_hits);
/* FmIndex::locate_many in its compact result form (texts shorter than 2^32 symbols, else GDX_ERR_UNSUPPORTED):
 * hit_counts[i] = number of hits of query i (nq entries; their prefix sums are the CSR offsets), hits as gdx_hit32 in
 * the same order as gdx_locate_many.  8 B per hit + 4 B per query cross PCIe instead of 16 + 8: locate is bound by
 * exactly those bytes end to end.  A host binding widens lazily while it iterates (the crate hands out
 * `Hit { usize, usize }` one at a time anyway, lib.rs:179-197).  Release with gdx_free_hits(idx, (gdx_hit *)hits). */
gdx_status gdx_locate_many_compact(const gdx_index *idx, const gdx_queries *queries, uint32_t *hit_counts,
                                   gdx_hit32 **hits, uint64_t *num_hits);
/* Cursor::locate / FmIndex::locate_interval (src/cursor.rs:71-73, src/lib.rs:187-197) for many
 * cursors at once. */
gdx_status gdx_locate_intervals(const gdx_index *idx, const uint64_t *starts, const uint64_t *ends,
                                uint64_t n, uint64_t *hit_offsets, gdx_hit **hits,
                                uint64_t *num_hits);
void gdx_free_hits(const gdx_index *idx, gdx_hit *hits);

/* ---- one batch over several replicas (SURVEY 8e; the drop-in for src/lib.rs:155-185 on a multi-GPU box) ---
 * The batch is cut into n_shards contiguous ranges (gdx_shard_range); this process owns the shards
 * [first_shard, first_shard + n_local) and searches shard first_shard + k on replicas[k], one host thread and
 * one pinned staging arena per GPU, no collective.  Results are written straight into the caller's arrays at
 * the queries' own positions (input order); entries of ranges owned by other processes are not touched.
 * Single process: first_shard = 0, n_local = n_shards = number of GPUs.  One process per GPU (MPI / torchrun):
 * n_local = 1, first_shard = rank, n_shards = world size. */
void gdx_shard_range(uint64_t n_items, uint32_t shard, uint32_t n_shards, uint64_t *begin, uint64_t *end);
gdx_status gdx_count_many_sharded(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                  uint32_t n_shards, const gdx_queries *queries, uint64_t *counts);
gdx_status gdx_cursors_many_sharded(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                    uint32_t n_shards, const gdx_queries *queries, uint64_t *starts,
                                    uint64_t *ends);
/* Hits come back per shard (no concatenation copy): shard_hits[k] (release with gdx_free_hits(replicas[k], ..))
 * holds the hits of local shard k, shard_first_hit[k] the number of hits of the local shards before it
 * (n_local + 1 entries).  hit_offsets (nq + 1 entries, the owned ranges and the entry after the last owned
 * query are written) index the concatenation of the local shards: the hits of query i of local shard k are
 * shard_hits[k][hit_offsets[i] - shard_first_hit[k] .. hit_offsets[i + 1] - shard_first_hit[k]). */
gdx_status gdx_locate_many_sharded(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                   uint32_t n_shards, const gdx_queries *queries, uint64_t *hit_offsets,
                                   gdx_hit **shard_hits, uint64_t *shard_first_hit);
/* compact form: hit_counts (nq entries, the owned ranges are written), per local shard its gdx_hit32 array and its
 * number of hits (n_local entries each); the hits of a shard's queries follow each other in query order */
gdx_status gdx_locate_many_sharded_compact(gdx_index *const *replicas, uint32_t n_local, uint32_t first_shard,
                                           uint32_t n_shards, const gdx_queries *queries, uint32_t *hit_counts,
                                           gdx_hit32 **shard_hits, uint64_t *shard_num_hits);
/* Cursor::extend_query_front (src/cursor.rs:34-51) for many cursors: in-place on starts/ends.  On an error
 * status the contents of pinned starts/ends are unspecified (the reference panics); pageable arrays are
 * left untouched. */
gdx_status gdx_extend_many(const gdx_index *idx, uint64_t *starts, uint64_t *ends,
                           const uint8_t *io_symbols, uint64_t n);

/* ---- approximate search, no counterpart in the reference -----------------------------------------
 * Hamming-distance search with up to max_mismatches substitutions, IO-byte batches (GDX_QUERIES_IO_BYTES) only.
 *   - A query of length m matches at text position p with d mismatches when the window [p, p + m) lies inside one
 *     text, every symbol of it is a searchable dense symbol, and it differs from the query in exactly d <= k
 *     positions, compared in the dense representation (case folding and ambiguity groups apply as everywhere else).
 *     A window holding `N`, another symbol that is not searchable or a sentinel never matches.
 *   - Every distinct matching window string is one non-empty SA interval [start, end); its mismatch count is its
 *     Hamming distance to the query.  The intervals of a query are pairwise disjoint and sorted by start.
 *   - k = 0 gives what gdx_cursors_many / gdx_count_many / gdx_locate_many give for a query of searchable symbols
 *     (no interval when that interval is empty).  The empty query gives [0, text_len) with 0 mismatches.
 *   - Errors are checked before any result is produced, and gdx_last_error_query() names the smallest offending
 *     query: a byte that is not a searchable symbol (not in the alphabet, or valid but not searchable such as `N`):
 *     GDX_ERR_INVALID_SYMBOL; a query longer than GDX_HAMMING_MAX_QUERY_LEN: GDX_ERR_UNSUPPORTED; offsets that
 *     decrease or leave the batch: GDX_ERR_BAD_ARG.  max_mismatches > GDX_HAMMING_MAX_MISMATCHES: GDX_ERR_BAD_ARG;
 *     GDX_QUERIES_PACKED_2BIT: GDX_ERR_UNSUPPORTED.  Results that do not fit into device memory: GDX_ERR_OOM
 *     (split the batch).  Nothing is truncated.
 *   - Results do not depend on the lookup depth, the storage type, the construction route, GDX_FLAG_NO_TEXT, the
 *     accelerators or gdx_index_set_text_verification.
 * gdx_stats: lf_steps counts search-node expansions (one per node that may still branch, one per exact LF pair). */
#define GDX_HAMMING_MAX_MISMATCHES 3
#define GDX_HAMMING_MAX_QUERY_LEN 256
typedef struct gdx_hamming_interval {
    uint64_t start, end;     /* SA interval of one matching window string */
    uint32_t mismatches;     /* its Hamming distance to the query */
    uint32_t reserved;       /* 0 */
} gdx_hamming_interval;

/* counts[i * (k + 1) + d] = occurrences of query i with exactly d mismatches */
gdx_status gdx_count_many_hamming(const gdx_index *idx, const gdx_queries *queries, uint32_t max_mismatches,
                                  uint64_t *counts);
/* CSR: the intervals of query i are intervals[interval_offsets[i] .. interval_offsets[i+1]), sorted by start;
 * interval_offsets has nq + 1 entries; library-allocated pinned memory, release with
 * gdx_free_hits(idx, (gdx_hit *)intervals) */
gdx_status gdx_cursors_many_hamming(const gdx_index *idx, const gdx_queries *queries, uint32_t max_mismatches,
                                    uint64_t *interval_offsets, gdx_hamming_interval **intervals,
                                    uint64_t *num_intervals);
/* CSR as gdx_locate_many; hits of a query in ascending SA-row order over all its intervals */
gdx_status gdx_locate_many_hamming(const gdx_index *idx, const gdx_queries *queries, uint32_t max_mismatches,
                                   uint64_t *hit_offsets, gdx_hit **hits, uint64_t *num_hits);

/* single-query forms (src/lib.rs:147-149,169-173,217-235); these follow the single-query code path
 * of the reference (the symbol left of an empty lookup interval is still translated). */
gdx_status gdx_cursor_for_query(const gdx_index *idx, const uint8_t *query, uint64_t len,
                                uint64_t *start, uint64_t *end);

/* ---- batched search with device-resident buffers (for pipelines that keep data in HBM) ---------
 * All pointers are device pointers on the index's device; `stream` is a cudaStream_t (NULL = the
 * legacy default stream).  Asynchronous: errors of the kernels are reported through *d_error
 * (device uint64: 0 = none, else 1 + index of the first offending query), which may be NULL. */
gdx_status gdx_cursors_many_device(const gdx_index *idx, const gdx_queries *d_queries,
                                   uint64_t *d_starts, uint64_t *d_ends, uint64_t *d_error,
                                   void *stream);
gdx_status gdx_count_many_device(const gdx_index *idx, const gdx_queries *d_queries,
                                 uint64_t *d_counts, uint64_t *d_error, void *stream);
/* locate rows [start,end) of n intervals whose CSR offsets are already known on the device */
gdx_status gdx_locate_intervals_device(const gdx_index *idx, const uint64_t *d_starts,
                                       const uint64_t *d_ends, uint64_t n,
                                       const uint64_t *d_hit_offsets, uint64_t num_hits,
                                       gdx_hit *d_hits, void *stream);

/* The staging thread pool (packing, copies between caller memory and pinned buffers) is created at first use
 * with GDX_HOST_THREADS threads, default: the CPUs the creating thread may run on, at most 32.  This call
 * re-creates it with `threads` threads (0 = the default rule, evaluated for the calling thread now); the new
 * workers inherit the caller's CPU affinity.  Must not run concurrently with searches.  Returns the new size. */
uint32_t gdx_host_pool_resize(uint32_t threads);
/* Tuning of the host packer (defaults: software prefetch 4096 bytes ahead, non-temporal stores of the packed words;
 * GDX_PACK_PREFETCH / GDX_PACK_STREAM set the same at start-up): for A/B measurements on a given host. */
void gdx_host_pack_tuning(int32_t prefetch_bytes, int32_t streaming_stores);

/* pinned host memory helpers (full-speed asynchronous H2D/D2H) */
gdx_status gdx_host_alloc(uint64_t bytes, void **out);
void gdx_host_free(void *p);

gdx_status gdx_get_stats(gdx_stats *out); /* thread local, last call */

/* measured random-gather ceiling of the device (SURVEY 8d): independent aligned `record_bytes`
 * loads at random offsets over a `table_bytes` table; returns GB/s of requested bytes.
 * chained != 0: the next two addresses of a thread depend on the data just loaded (the access
 * pattern of an LF step) instead of on a counter. */
gdx_status gdx_measure_random_gather(int32_t device, uint64_t table_bytes, uint32_t record_bytes,
                                     uint64_t loads, int32_t chained, double *gbps_out,
                                     double *gloads_out);

#ifdef __cplusplus
}
#endif
#endif /* GENEDEX_B200_H */
