/*
 * dach_oracle.h -- CPU ORACLE for the daachorse scan path.  TEST INFRASTRUCTURE ONLY.
 *
 * This is a plain-C restatement of the reference crate daac-tools/daachorse 4.0.0
 * (construction, wire format and the per-byte / per-char scan loops).  It exists to
 * check the CUDA product path; nothing under daachorse_b200/ may include, link or
 * call it.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs use it.
 *
 * Parity pinning: the Rust crate cannot be compiled in this environment (no rustc),
 * so this oracle is pinned against the reference's own fixtures instead (see
 * tests/test_oracle_golden.py): the 136 SearchTest vectors of
 * tests/aho_corasick_crate_test.rs:63-382 under the 12 configurations at :537-645,
 * the BASE/CHECK/FAIL layout goldens (src/bytewise.rs:1257-1309,
 * src/charwise.rs:1214-1266), the test_n_blocks_* layouts, the heap_bytes /
 * num_states doc constants, the charwise zero-length multibyte vectors, the UTF-8
 * decoder table, the mapper ranks and the serializer LE goldens.
 *
 * All file:line citations are relative to the daachorse 4.0.0 repository.
 */
#ifndef DACH_ORACLE_H
#define DACH_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* src/errors.rs:10-22 (+ the match-kind assert of src/bytewise.rs:194-197) */
enum {
    ORC_OK = 0,
    ORC_INVALID_ARGUMENT = 1,
    ORC_AUTOMATON_SCALE = 2,
    ORC_INVALID_CONVERSION = 3,
    ORC_INVALID_AUTOMATON = 4,
    ORC_MATCH_KIND_MISMATCH = 5
};

/* src/lib.rs:324-346 */
enum { ORC_STANDARD = 0, ORC_LEFTMOST_LONGEST = 1, ORC_LEFTMOST_FIRST = 2 };

/* scan modes (iterators of src/bytewise/iter.rs, src/charwise/iter.rs) */
enum {
    ORC_FIND = 0,                       /* FindIterator */
    ORC_FIND_OVERLAPPING = 1,           /* FindOverlappingIterator */
    ORC_FIND_OVERLAPPING_NO_SUFFIX = 2, /* FindOverlappingNoSuffixIterator */
    ORC_LEFTMOST_FIND = 3,              /* LeftmostFindIterator */
    ORC_FIND_STEPPER = 4,               /* FindStepper driven as in tests/aho_corasick_crate_test.rs:422-463 */
    ORC_FIND_OVERLAPPING_STEPPER = 5    /* FindOverlappingStepper, ibid. :477-520 */
};

/* Match reported as (start, end, value); start = end - length (src/lib.rs:301-303) */
typedef struct {
    uint32_t start, end, value;
} orc_match;

typedef struct orc_pma orc_pma;

/* Construction: patterns are given as one byte blob + n+1 offsets; values == NULL means
 * value i for pattern i (builder.rs:152-167).  charwise != 0 builds the
 * CharwiseDoubleArrayAhoCorasick (patterns must be valid UTF-8). */
int orc_build(int charwise, const uint8_t *bytes, const uint64_t *offs, const uint32_t *values,
              uint32_t n, uint8_t match_kind, uint32_t num_free_blocks, orc_pma **out);
void orc_free(orc_pma *p);

/* Wire format (src/bytewise.rs:801-820, src/charwise.rs:831-848). */
size_t orc_serialized_bytes(const orc_pma *p);
size_t orc_serialize(const orc_pma *p, uint8_t *dst, size_t cap);
int orc_deserialize(int charwise, const uint8_t *src, size_t len, orc_pma **out, size_t *consumed);

/* Introspection. */
int orc_is_charwise(const orc_pma *p);
uint8_t orc_match_kind(const orc_pma *p);
uint32_t orc_num_states(const orc_pma *p);
size_t orc_heap_bytes(const orc_pma *p);
size_t orc_num_elements(const orc_pma *p); /* length of the double array */
size_t orc_num_outputs(const orc_pma *p);
uint32_t orc_max_pattern_len(const orc_pma *p); /* max Output.length */
/* layout peek for the golden-layout tests: returns 0 on success */
int orc_peek_state(const orc_pma *p, size_t idx, uint32_t *base, uint32_t *check, uint32_t *fail,
                   uint32_t *output_pos);
uint32_t orc_mapper_get(const orc_pma *p, uint32_t code_point); /* UINT32_MAX = None */
uint32_t orc_alphabet_size(const orc_pma *p);

/* One haystack.  Returns ORC_OK / ORC_MATCH_KIND_MISMATCH; *n_out receives the number
 * of matches the iterator yields (even when it exceeds cap; only the first cap are
 * written). */
int orc_scan(const orc_pma *p, int mode, const uint8_t *hay, size_t len, orc_match *out, size_t cap,
             size_t *n_out);

/* UTF-8 decoder table test hook (src/charwise/iter.rs:71-97): decodes one char at
 * hay[*pos], advances *pos to its end offset, returns the code point. */
uint32_t orc_utf8_next(const uint8_t *hay, size_t *pos);

/* Batch over n haystacks (text blob + n+1 offsets), nthreads host threads over
 * contiguous haystack ranges.  counts[i] = matches of haystack i; hashes[i] (optional)
 * = order-sensitive 64-bit hash of its tuples; if out != NULL the tuples are written
 * densely in haystack order (two passes) and out_cap bounds them.  Returns ORC_OK or an
 * error; *total receives the total match count. */
int orc_scan_batch(const orc_pma *p, int mode, const uint8_t *text, const uint64_t *offs, uint64_t n,
                   int nthreads, uint64_t *counts, uint64_t *hashes, orc_match *out, uint64_t out_cap,
                   uint64_t *total);

/* The timed CPU baseline of bench.py: same scan loops, on the crate's array-of-structs record layout, on a
 * persistent pool of threads pinned to the CPUs the process may use, every match stored into a per-thread
 * ring (a consumer collecting them), no checker hash.  counts may be NULL. */
int orc_bench_batch(const orc_pma *p, int mode, const uint8_t *text, const uint64_t *offs, uint64_t n, int nthreads,
                    uint64_t *counts, uint64_t *total);

/* The order-sensitive tuple hash used by orc_scan_batch (also implemented on the
 * Python side and on the GPU side for full-size parity). */
uint64_t orc_hash_step(uint64_t h, uint32_t start, uint32_t end, uint32_t value);
/* per-haystack hashes (as orc_scan_batch's `hashes`) of an existing result: matches + n+1 offsets */
void orc_hash_matches(const orc_match *m, const uint64_t *offs, uint64_t n, uint64_t *hashes);

#ifdef __cplusplus
}
#endif
#endif
