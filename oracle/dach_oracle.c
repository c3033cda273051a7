/*
 * dach_oracle.c -- CPU ORACLE (test infrastructure only; see dach_oracle.h).
 *
 * Plain-C restatement of daac-tools/daachorse 4.0.0.  Each function cites the
 * reference file:line (relative to the daachorse 4.0.0 repository) whose control flow it follows.
 * V (the pattern value type) is fixed to u32.
 */
#define _GNU_SOURCE
#include "dach_oracle.h"

#include <pthread.h>
#include <sched.h>
#include <stdlib.h>
#include <string.h>

#define ROOT 0u /* src/nfa_builder.rs:12, src/bytewise.rs:25, src/charwise.rs */
#define DEAD 1u /* src/nfa_builder.rs:14, src/bytewise.rs:27 */
#define NONE32 0xffffffffu
#define U24_MAX 0x00ffffffu     /* src/intpack.rs:15 */
#define INVALID_CODE 0xffffffffu /* src/charwise/mapper.rs:7 */

/* ------------------------------------------------------------------------- */
/* Sparse NFA (src/nfa_builder.rs, src/edge_map.rs)                            */
/* ------------------------------------------------------------------------- */

typedef struct {
    uint32_t label, child;
} edge_t;

typedef struct {
    /* EdgeMap: Empty / One / Many(sorted by label)  (src/edge_map.rs:4-9) */
    uint32_t n_edges, cap_edges;
    edge_t one;
    edge_t *many;
    uint32_t fail;       /* Cell<u32>, default ROOT (nfa_builder.rs:45) */
    uint32_t pend_head;  /* this state's own (value,length) list, newest first */
    uint32_t output_pos; /* Option<NonZeroU32>, 0 = None */
} nfa_state;

typedef struct {
    uint32_t value, length, next;
} pend_t;

typedef struct {
    uint32_t value, length, parent; /* src/lib.rs:213-218, parent 0 = None */
} output_t;

typedef struct {
    nfa_state *states;
    size_t n_states, cap_states;
    pend_t *pend;
    size_t n_pend, cap_pend;
    output_t *outputs;
    size_t n_outputs, cap_outputs;
    size_t len; /* number of registered patterns (nfa_builder.rs:111) */
    uint8_t match_kind;
} nfa_t;

static void *xrealloc(void *p, size_t n) {
    void *q = realloc(p, n ? n : 1);
    if (!q) abort();
    return q;
}

static const edge_t *edges_of(const nfa_state *s) { return s->n_edges <= 1 ? &s->one : s->many; }

static void nfa_push_state(nfa_t *nfa) {
    if (nfa->n_states == nfa->cap_states) {
        nfa->cap_states = nfa->cap_states ? nfa->cap_states * 2 : 1024;
        nfa->states = (nfa_state *)xrealloc(nfa->states, nfa->cap_states * sizeof(nfa_state));
    }
    nfa_state *s = &nfa->states[nfa->n_states++];
    memset(s, 0, sizeof(*s));
    s->fail = ROOT;
    s->pend_head = NONE32;
    s->output_pos = 0;
}

/* nfa_builder.rs:65-75 */
static void nfa_init(nfa_t *nfa, uint8_t match_kind) {
    memset(nfa, 0, sizeof(*nfa));
    nfa->match_kind = match_kind;
    nfa_push_state(nfa); /* root */
    nfa_push_state(nfa); /* dead */
}

static void nfa_destroy(nfa_t *nfa) {
    for (size_t i = 0; i < nfa->n_states; i++)
        if (nfa->states[i].many) free(nfa->states[i].many);
    free(nfa->states);
    free(nfa->pend);
    free(nfa->outputs);
    memset(nfa, 0, sizeof(*nfa));
}

/* EdgeMap::get (edge_map.rs:46-55); returns NONE32 when absent. */
static uint32_t nfa_child(const nfa_t *nfa, uint32_t state_id, uint32_t c) {
    const nfa_state *s = &nfa->states[state_id];
    if (s->n_edges == 0) return NONE32;
    if (s->n_edges == 1) return s->one.label == c ? s->one.child : NONE32;
    size_t lo = 0, hi = s->n_edges;
    while (lo < hi) {
        size_t mid = (lo + hi) / 2;
        if (s->many[mid].label < c)
            lo = mid + 1;
        else
            hi = mid;
    }
    if (lo < s->n_edges && s->many[lo].label == c) return s->many[lo].child;
    return NONE32;
}

/* EdgeMap::insert for a key known to be absent (edge_map.rs:15-44): keeps label order. */
static void nfa_insert_edge(nfa_t *nfa, uint32_t state_id, uint32_t c, uint32_t child) {
    nfa_state *s = &nfa->states[state_id];
    if (s->n_edges == 0) {
        s->one.label = c;
        s->one.child = child;
        s->n_edges = 1;
        return;
    }
    if (s->n_edges == 1) {
        s->cap_edges = 4;
        s->many = (edge_t *)xrealloc(NULL, s->cap_edges * sizeof(edge_t));
        if (c < s->one.label) {
            s->many[0].label = c;
            s->many[0].child = child;
            s->many[1] = s->one;
        } else {
            s->many[0] = s->one;
            s->many[1].label = c;
            s->many[1].child = child;
        }
        s->n_edges = 2;
        return;
    }
    if (s->n_edges == s->cap_edges) {
        s->cap_edges *= 2;
        s->many = (edge_t *)xrealloc(s->many, s->cap_edges * sizeof(edge_t));
    }
    size_t pos = s->n_edges;
    while (pos > 0 && s->many[pos - 1].label > c) {
        s->many[pos] = s->many[pos - 1];
        pos--;
    }
    s->many[pos].label = c;
    s->many[pos].child = child;
    s->n_edges++;
}

/* NfaBuilder::add (nfa_builder.rs:78-113).  pattern_len = byte length of the pattern. */
static int nfa_add(nfa_t *nfa, const uint32_t *labels, size_t n_labels, uint64_t pattern_len,
                   uint32_t value) {
    if (pattern_len > 0xffffffffull) return ORC_INVALID_ARGUMENT; /* :79-83 */
    uint32_t state_id = ROOT;
    for (size_t i = 0; i < n_labels; i++) {
        uint32_t c = labels[i];
        if (nfa->match_kind == ORC_LEFTMOST_FIRST) {
            /* :87-92 the descendants of an output state are never searched */
            if (nfa->states[state_id].pend_head != NONE32) return ORC_OK;
        }
        uint32_t next = nfa_child(nfa, state_id, c);
        if (next != NONE32) {
            state_id = next;
        } else if (nfa->n_states <= 0xffffffffull) { /* :96 u32::try_from(states.len()) */
            uint32_t nid = (uint32_t)nfa->n_states;
            nfa_insert_edge(nfa, state_id, c, nid);
            nfa_push_state(nfa);
            state_id = nid;
        } else {
            return ORC_AUTOMATON_SCALE;
        }
    }
    /* :107-109 push (value, pattern_len); list is kept newest-first */
    if (nfa->n_pend == nfa->cap_pend) {
        nfa->cap_pend = nfa->cap_pend ? nfa->cap_pend * 2 : 1024;
        nfa->pend = (pend_t *)xrealloc(nfa->pend, nfa->cap_pend * sizeof(pend_t));
    }
    pend_t *pe = &nfa->pend[nfa->n_pend];
    pe->value = value;
    pe->length = (uint32_t)pattern_len;
    pe->next = nfa->states[state_id].pend_head;
    nfa->states[state_id].pend_head = (uint32_t)nfa->n_pend;
    nfa->n_pend++;
    nfa->len++;
    return ORC_OK;
}

/* NfaBuilder::build_fails (nfa_builder.rs:115-144).  Returns the BFS order q. */
static uint32_t *nfa_build_fails(nfa_t *nfa, size_t *q_len) {
    uint32_t *q = (uint32_t *)xrealloc(NULL, nfa->n_states * sizeof(uint32_t));
    size_t qn = 0;
    {
        const nfa_state *r = &nfa->states[ROOT];
        const edge_t *e = edges_of(r);
        for (uint32_t i = 0; i < r->n_edges; i++) q[qn++] = e[i].child;
    }
    size_t qi = 0;
    while (qi < qn) {
        uint32_t state_id = q[qi++];
        const nfa_state *s = &nfa->states[state_id];
        const edge_t *e = edges_of(s);
        for (uint32_t i = 0; i < s->n_edges; i++) {
            uint32_t c = e[i].label, child_id = e[i].child;
            uint32_t fail_id = s->fail, new_fail;
            for (;;) {
                uint32_t cf = nfa_child(nfa, fail_id, c);
                if (cf != NONE32) {
                    new_fail = cf;
                    break;
                }
                uint32_t next_fail = nfa->states[fail_id].fail;
                if (fail_id == ROOT && next_fail == ROOT) {
                    new_fail = ROOT;
                    break;
                }
                fail_id = next_fail;
            }
            nfa->states[child_id].fail = new_fail;
            q[qn++] = child_id;
        }
    }
    *q_len = qn;
    return q;
}

/* NfaBuilder::build_fails_leftmost (nfa_builder.rs:146-201). */
static uint32_t *nfa_build_fails_leftmost(nfa_t *nfa, size_t *q_len) {
    uint32_t *q = (uint32_t *)xrealloc(NULL, nfa->n_states * sizeof(uint32_t));
    size_t qn = 0;
    {
        const nfa_state *r = &nfa->states[ROOT];
        const edge_t *e = edges_of(r);
        for (uint32_t i = 0; i < r->n_edges; i++) q[qn++] = e[i].child;
        if (r->pend_head != NONE32) { /* :151-160 */
            for (uint32_t i = 0; i < r->n_edges; i++) nfa->states[e[i].child].fail = DEAD;
        }
    }
    size_t qi = 0;
    while (qi < qn) {
        uint32_t state_id = q[qi++];
        nfa_state *s = &nfa->states[state_id];
        if (s->pend_head != NONE32) s->fail = DEAD; /* :169-172 */
        const edge_t *e = edges_of(s);
        for (uint32_t i = 0; i < s->n_edges; i++) {
            uint32_t c = e[i].label, child_id = e[i].child;
            uint32_t fail_id = s->fail, new_fail;
            if (fail_id == DEAD) { /* :177-179 */
                new_fail = DEAD;
            } else {
                for (;;) {
                    uint32_t cf = nfa_child(nfa, fail_id, c);
                    if (cf != NONE32) {
                        new_fail = cf;
                        break;
                    }
                    uint32_t next_fail = nfa->states[fail_id].fail;
                    if (next_fail == DEAD) {
                        new_fail = DEAD;
                        break;
                    }
                    if (fail_id == ROOT && next_fail == ROOT) {
                        new_fail = ROOT;
                        break;
                    }
                    fail_id = next_fail;
                }
            }
            nfa->states[child_id].fail = new_fail;
            q[qn++] = child_id;
        }
    }
    *q_len = qn;
    return q;
}

static void nfa_push_output(nfa_t *nfa, uint32_t value, uint32_t length, uint32_t parent) {
    if (nfa->n_outputs == nfa->cap_outputs) {
        nfa->cap_outputs = nfa->cap_outputs ? nfa->cap_outputs * 2 : 1024;
        nfa->outputs = (output_t *)xrealloc(nfa->outputs, nfa->cap_outputs * sizeof(output_t));
    }
    output_t *o = &nfa->outputs[nfa->n_outputs++];
    o->value = value;
    o->length = length;
    o->parent = parent;
}

/* NfaBuilder::build_outputs (nfa_builder.rs:203-222). */
static void nfa_build_outputs(nfa_t *nfa, const uint32_t *q, size_t q_len) {
    {
        nfa_state *s = &nfa->states[ROOT];
        uint32_t last_pos = 0;
        for (uint32_t pi = s->pend_head; pi != NONE32; pi = nfa->pend[pi].next) { /* .rev() */
            nfa_push_output(nfa, nfa->pend[pi].value, nfa->pend[pi].length, last_pos);
            last_pos = (uint32_t)nfa->n_outputs;
        }
        s->output_pos = last_pos;
    }
    for (size_t k = 0; k < q_len; k++) {
        nfa_state *s = &nfa->states[q[k]];
        uint32_t last_pos = nfa->states[s->fail].output_pos;
        for (uint32_t pi = s->pend_head; pi != NONE32; pi = nfa->pend[pi].next) {
            nfa_push_output(nfa, nfa->pend[pi].value, nfa->pend[pi].length, last_pos);
            last_pos = (uint32_t)nfa->n_outputs;
        }
        s->output_pos = last_pos;
    }
}

/* ------------------------------------------------------------------------- */
/* BuildHelper (src/build_helper.rs)                                           */
/* ------------------------------------------------------------------------- */

typedef struct {
    uint32_t *next, *prev;
    uint8_t *used_base, *used_index;
    uint32_t block_len, num_free_blocks, num_blocks, capacity;
    int has_head;
    uint32_t head;
} helper_t;

/* BuildHelper::new (build_helper.rs:30-44) */
static int helper_init(helper_t *h, uint32_t block_len, uint32_t num_free_blocks) {
    memset(h, 0, sizeof(*h));
    uint64_t cap = (uint64_t)block_len * (uint64_t)num_free_blocks;
    if (cap > 0xffffffffull) return ORC_AUTOMATON_SCALE; /* checked_mul */
    if (cap == 0) abort();                               /* assert_ne!(capacity, 0) */
    h->capacity = (uint32_t)cap;
    h->block_len = block_len;
    h->num_free_blocks = num_free_blocks;
    h->next = (uint32_t *)calloc(cap, sizeof(uint32_t));
    h->prev = (uint32_t *)calloc(cap, sizeof(uint32_t));
    h->used_base = (uint8_t *)calloc(cap, 1);
    h->used_index = (uint8_t *)calloc(cap, 1);
    if (!h->next || !h->prev || !h->used_base || !h->used_index) abort();
    return ORC_OK;
}

static void helper_destroy(helper_t *h) {
    free(h->next);
    free(h->prev);
    free(h->used_base);
    free(h->used_index);
}

static uint32_t helper_num_elements(const helper_t *h) { return h->num_blocks * h->block_len; }
/* active_block_range (build_helper.rs:61-63) */
static uint32_t helper_active_block_start(const helper_t *h) {
    return h->num_blocks > h->num_free_blocks ? h->num_blocks - h->num_free_blocks : 0;
}
/* offset (build_helper.rs:203-207): index must be inside the active range */
static uint32_t helper_off(const helper_t *h, uint32_t idx) {
    uint32_t lo = helper_active_block_start(h) * h->block_len;
    uint32_t hi = h->num_blocks * h->block_len;
    if (!(idx >= lo && idx < hi)) abort();
    return idx % h->capacity;
}
static int helper_is_used_base(const helper_t *h, uint32_t b) { return h->used_base[helper_off(h, b)]; }
static int helper_is_used_index(const helper_t *h, uint32_t i) { return h->used_index[helper_off(h, i)]; }
static void helper_use_base(helper_t *h, uint32_t b) { h->used_base[helper_off(h, b)] = 1; }

/* use_index (build_helper.rs:118-130) */
static void helper_use_index(helper_t *h, uint32_t idx) {
    uint32_t o = helper_off(h, idx);
    h->used_index[o] = 1;
    uint32_t next = h->next[o], prev = h->prev[o];
    h->next[helper_off(h, prev)] = next;
    h->prev[helper_off(h, next)] = prev;
    if (!h->has_head) abort(); /* head_idx.unwrap() */
    if (h->head == idx) {
        if (next != idx) {
            h->head = next;
        } else {
            h->has_head = 0;
        }
    }
}

/* dropped_block (build_helper.rs:177-179): returns 1 and the block index if a block drops */
static int helper_dropped_block(const helper_t *h, uint32_t *blk) {
    if (h->capacity <= helper_num_elements(h)) {
        *blk = helper_active_block_start(h);
        return 1;
    }
    return 0;
}

/* push_block (build_helper.rs:133-173) */
static int helper_push_block(helper_t *h) {
    if (helper_num_elements(h) > 0xffffffffu - h->block_len) return ORC_AUTOMATON_SCALE;
    uint32_t closed;
    if (helper_dropped_block(h, &closed)) {
        uint32_t end_idx = (closed + 1) * h->block_len;
        while (h->has_head) {
            if (end_idx <= h->head) break;
            helper_use_index(h, h->head);
        }
    }
    uint32_t old_len = helper_num_elements(h);
    uint32_t new_len = old_len + h->block_len;
    h->num_blocks += 1;
    for (uint32_t idx = old_len; idx < new_len; idx++) {
        uint32_t o = helper_off(h, idx);
        h->used_base[o] = 0;
        h->used_index[o] = 0;
        h->next[o] = idx + 1;
        h->prev[o] = idx - 1; /* wrapping_sub */
    }
    if (h->has_head) {
        uint32_t head = h->head;
        uint32_t tail = h->prev[helper_off(h, head)];
        h->prev[helper_off(h, old_len)] = tail;
        h->next[helper_off(h, tail)] = old_len;
        h->next[helper_off(h, new_len - 1)] = head;
        h->prev[helper_off(h, head)] = new_len - 1;
    } else {
        h->prev[helper_off(h, old_len)] = new_len - 1;
        h->next[helper_off(h, new_len - 1)] = old_len;
        h->has_head = 1;
        h->head = old_len;
    }
    return ORC_OK;
}

/* unused_base_in_block (build_helper.rs:76-80): lowest unused base, NONE32 if none */
static uint32_t helper_unused_base_in_block(const helper_t *h, uint32_t block_idx) {
    uint32_t start = block_idx * h->block_len, end = start + h->block_len;
    for (uint32_t b = start; b < end; b++)
        if (!helper_is_used_base(h, b)) return b;
    return NONE32;
}

/* ------------------------------------------------------------------------- */
/* The automaton                                                               */
/* ------------------------------------------------------------------------- */

struct orc_pma {
    int charwise;
    uint8_t match_kind;
    uint32_t num_states;
    /* double array; n_slots entries.  Bytewise: base, fail, opos_ch (src/bytewise.rs:1131-1137);
     * a leftmost bytewise automaton keeps base/opos_ch in "leftmost_states" and fail in "fails"
     * (src/bytewise.rs:61-63) -- same three arrays here, flagged by match_kind.
     * Charwise: base, check, fail, output_pos (src/charwise.rs:1096-1101). */
    size_t n_slots;
    uint32_t *base, *fail;
    uint32_t *opos_ch;            /* bytewise */
    uint32_t *check, *output_pos; /* charwise */
    uint32_t root_table[256];     /* bytewise Standard (src/bytewise.rs:1040-1056) */
    int has_root_table;
    /* CodeMapper (src/charwise/mapper.rs:10-13) */
    uint32_t *table;
    size_t table_len;
    uint32_t alphabet_size;
    output_t *outputs;
    size_t n_outputs;
    /* The crate's in-memory records, one array of structs each -- what its scan loops actually walk:
     *   bytewise Standard  State<u32>{base, fail, opos_ch}      12 B  (src/bytewise.rs:1131-1137)
     *   bytewise leftmost  State<Empty>{base, opos_ch} 8 B + fails[] 4 B  (src/bytewise.rs:61-63)
     *   charwise           State{base, check, fail, output_pos} 16 B  (src/charwise.rs:1096-1101)
     * Built from the arrays above when construction / deserialisation ends; every scan below reads these,
     * so that the CPU baseline timed with this file pays one cache line per visited state like the crate
     * does (VERDICT r1: three parallel arrays cost up to three). */
    struct bw_state *st12;
    struct lm_state *st8;
    struct cw_state *st16;
};
struct bw_state {
    uint32_t base, fail, opos_ch;
};
struct lm_state {
    uint32_t base, opos_ch;
};
struct cw_state {
    uint32_t base, check, fail, output_pos;
};

static void build_scan_records(orc_pma *p) {
    const size_t n = p->n_slots;
    free(p->st12), free(p->st8), free(p->st16);
    p->st12 = NULL, p->st8 = NULL, p->st16 = NULL;
    if (p->charwise) {
        p->st16 = (struct cw_state *)xrealloc(NULL, (n ? n : 1) * sizeof(struct cw_state));
        for (size_t i = 0; i < n; i++) {
            p->st16[i].base = p->base[i];
            p->st16[i].check = p->check[i];
            p->st16[i].fail = p->fail[i];
            p->st16[i].output_pos = p->output_pos[i];
        }
    } else if (p->match_kind == ORC_LEFTMOST_LONGEST || p->match_kind == ORC_LEFTMOST_FIRST) {
        p->st8 = (struct lm_state *)xrealloc(NULL, (n ? n : 1) * sizeof(struct lm_state));
        for (size_t i = 0; i < n; i++) {
            p->st8[i].base = p->base[i];
            p->st8[i].opos_ch = p->opos_ch[i];
        }
    } else {
        p->st12 = (struct bw_state *)xrealloc(NULL, (n ? n : 1) * sizeof(struct bw_state));
        for (size_t i = 0; i < n; i++) {
            p->st12[i].base = p->base[i];
            p->st12[i].fail = p->fail[i];
            p->st12[i].opos_ch = p->opos_ch[i];
        }
    }
}

void orc_free(orc_pma *p) {
    if (!p) return;
    free(p->base);
    free(p->fail);
    free(p->opos_ch);
    free(p->check);
    free(p->output_pos);
    free(p->table);
    free(p->outputs);
    free(p->st12);
    free(p->st8);
    free(p->st16);
    free(p);
}

static int is_leftmost(uint8_t k) { return k == ORC_LEFTMOST_LONGEST || k == ORC_LEFTMOST_FIRST; }

/* build_root_table (src/bytewise.rs:1040-1056) */
static void build_root_table(orc_pma *p) {
    for (int c = 0; c < 256; c++) p->root_table[c] = ROOT;
    if (p->n_slots > 0 && p->base[ROOT] != 0) {
        uint32_t b = p->base[ROOT];
        for (uint32_t c = 0; c < 256; c++) {
            uint32_t child = b ^ c;
            if (child < p->n_slots && (p->opos_ch[child] & 0xff) == c) p->root_table[c] = child;
        }
    }
    p->has_root_table = 1;
}

/* ---- bytewise double-array construction (src/bytewise/builder.rs) -------- */

typedef struct {
    orc_pma *p;
    size_t cap_slots;
} bw_builder;

static void bw_resize(bw_builder *b, size_t n) {
    orc_pma *p = b->p;
    if (n > b->cap_slots) {
        size_t nc = b->cap_slots ? b->cap_slots : 256;
        while (nc < n) nc *= 2;
        p->base = (uint32_t *)xrealloc(p->base, nc * 4);
        p->fail = (uint32_t *)xrealloc(p->fail, nc * 4);
        p->opos_ch = (uint32_t *)xrealloc(p->opos_ch, nc * 4);
        b->cap_slots = nc;
    }
    for (size_t i = p->n_slots; i < n; i++) { /* State::default(): all zero */
        p->base[i] = 0;
        p->fail[i] = 0;
        p->opos_ch[i] = 0;
    }
    p->n_slots = n;
}

static void bw_set_check(orc_pma *p, uint32_t idx, uint32_t c) {
    p->opos_ch[idx] = (p->opos_ch[idx] & 0xffffff00u) | (c & 0xff); /* intpack.rs:51-53 */
}

/* remove_invalid_checks (builder.rs:391-400) */
static void bw_remove_invalid_checks(orc_pma *p, uint32_t block_idx, const helper_t *h) {
    uint32_t ub = helper_unused_base_in_block(h, block_idx);
    if (ub == NONE32) return;
    for (uint32_t c = 0; c < 256; c++) {
        uint32_t idx = ub ^ c;
        if (idx == ROOT || idx == DEAD || !helper_is_used_index(h, idx)) bw_set_check(p, idx, c);
    }
}

/* extend_array (builder.rs:372-388) */
static int bw_extend_array(bw_builder *b, helper_t *h) {
    if (b->p->n_slots > (size_t)(0xffffffffu - 256u)) return ORC_AUTOMATON_SCALE;
    uint32_t closed;
    if (helper_dropped_block(h, &closed)) bw_remove_invalid_checks(b->p, closed, h);
    int rc = helper_push_block(h);
    if (rc) return rc;
    bw_resize(b, b->p->n_slots + 256);
    return ORC_OK;
}

/* find_base + check_valid_base (builder.rs:347-370) */
static uint32_t bw_find_base(const orc_pma *p, const helper_t *h, const uint32_t *labels, size_t nl) {
    if (h->has_head) {
        uint32_t idx = h->head;
        for (;;) {
            uint32_t base = idx ^ labels[0];
            int ok = !helper_is_used_base(h, base);
            for (size_t i = 0; ok && i < nl; i++)
                if (helper_is_used_index(h, base ^ labels[i])) ok = 0;
            if (ok && base != 0) return base; /* NonZeroU32::new(base) */
            /* VacantIter::next (build_helper.rs:219-226) */
            uint32_t next = h->next[helper_off(h, idx)];
            if (next == h->head) break;
            idx = next;
        }
    }
    return (uint32_t)p->n_slots;
}

static int bw_build_double_array(orc_pma *p, const nfa_t *nfa, uint32_t num_free_blocks) {
    bw_builder b = {p, 0};
    helper_t h;
    /* init_array (builder.rs:336-344) */
    bw_resize(&b, 256);
    int rc = helper_init(&h, 256, num_free_blocks);
    if (rc) return rc;
    rc = helper_push_block(&h);
    if (rc) abort(); /* .unwrap() */
    helper_use_index(&h, ROOT);
    helper_use_index(&h, DEAD);

    size_t ns = nfa->n_states;
    uint32_t *map = (uint32_t *)xrealloc(NULL, ns * 4);
    for (size_t i = 0; i < ns; i++) map[i] = DEAD;
    map[ROOT] = ROOT;
    uint32_t *stack = (uint32_t *)xrealloc(NULL, (ns + 1) * 4);
    size_t sp = 0;
    stack[sp++] = ROOT;
    uint32_t labels[256];

    /* builder.rs:277-305 */
    while (sp > 0) {
        uint32_t state_id = stack[--sp];
        const nfa_state *s = &nfa->states[state_id];
        uint32_t state_idx = map[state_id];
        if (s->n_edges == 0) continue;
        const edge_t *e = edges_of(s);
        for (uint32_t i = 0; i < s->n_edges; i++) labels[i] = e[i].label;
        uint32_t base = bw_find_base(p, &h, labels, s->n_edges);
        if ((size_t)base >= p->n_slots) {
            rc = bw_extend_array(&b, &h);
            if (rc) goto done;
        }
        for (uint32_t i = 0; i < s->n_edges; i++) {
            uint32_t child_idx = base ^ e[i].label;
            helper_use_index(&h, child_idx);
            bw_set_check(p, child_idx, e[i].label);
            map[e[i].child] = child_idx;
            stack[sp++] = e[i].child;
        }
        p->base[state_idx] = base;
        helper_use_base(&h, base);
    }

    /* builder.rs:308-326: fail & output_pos */
    for (size_t i = 0; i < ns; i++) {
        if (i == DEAD) continue;
        uint32_t idx = map[i];
        uint32_t opos = nfa->states[i].output_pos;
        if (opos > U24_MAX) { /* set_output_pos (src/bytewise.rs:1179-1187) */
            rc = ORC_AUTOMATON_SCALE;
            goto done;
        }
        p->opos_ch[idx] = (opos << 8) | (p->opos_ch[idx] & 0xff);
        uint32_t fail_id = nfa->states[i].fail;
        p->fail[idx] = fail_id == DEAD ? DEAD : map[fail_id];
    }
    /* builder.rs:328-330 */
    for (uint32_t blk = helper_active_block_start(&h); blk < h.num_blocks; blk++)
        bw_remove_invalid_checks(p, blk, &h);
    rc = ORC_OK;
done:
    free(map);
    free(stack);
    helper_destroy(&h);
    return rc;
}

/* ---- charwise construction (src/charwise/builder.rs, mapper.rs) ----------- */

typedef struct {
    uint32_t c, f;
} cf_t;

/* mapper.rs:23: frequency descending, then code point ascending */
static int cf_cmp(const void *a, const void *b) {
    const cf_t *x = (const cf_t *)a, *y = (const cf_t *)b;
    if (x->f != y->f) return x->f > y->f ? -1 : 1;
    if (x->c != y->c) return x->c < y->c ? -1 : 1;
    return 0;
}

/* CodeMapper::new (mapper.rs:16-34) */
static void mapper_new(orc_pma *p, const uint32_t *freqs, size_t n) {
    cf_t *sorted = (cf_t *)xrealloc(NULL, (n ? n : 1) * sizeof(cf_t));
    size_t m = 0;
    for (size_t c = 0; c < n; c++)
        if (freqs[c] != 0) {
            sorted[m].c = (uint32_t)c;
            sorted[m].f = freqs[c];
            m++;
        }
    qsort(sorted, m, sizeof(cf_t), cf_cmp);
    p->table = (uint32_t *)xrealloc(NULL, (n ? n : 1) * 4);
    p->table_len = n;
    for (size_t c = 0; c < n; c++) p->table[c] = INVALID_CODE;
    for (size_t i = 0; i < m; i++) p->table[sorted[i].c] = (uint32_t)i;
    p->alphabet_size = (uint32_t)m;
    free(sorted);
}

/* CodeMapper::get (mapper.rs:36-42): INVALID_CODE stands for None */
static inline uint32_t mapper_get(const orc_pma *p, uint32_t c) {
    if ((size_t)c >= p->table_len) return INVALID_CODE;
    return p->table[c];
}

static uint32_t next_pow2_u32(uint32_t x) { /* u32::next_power_of_two; 0 -> 1 */
    uint32_t r = 1;
    while (r < x) r <<= 1;
    return r;
}

typedef struct {
    orc_pma *p;
    size_t cap_slots;
} cw_builder;

static void cw_resize(cw_builder *b, size_t n) {
    orc_pma *p = b->p;
    if (n > b->cap_slots) {
        size_t nc = b->cap_slots ? b->cap_slots : 256;
        while (nc < n) nc *= 2;
        p->base = (uint32_t *)xrealloc(p->base, nc * 4);
        p->check = (uint32_t *)xrealloc(p->check, nc * 4);
        p->fail = (uint32_t *)xrealloc(p->fail, nc * 4);
        p->output_pos = (uint32_t *)xrealloc(p->output_pos, nc * 4);
        b->cap_slots = nc;
    }
    for (size_t i = p->n_slots; i < n; i++) { /* State::default (src/charwise.rs:1103-1112) */
        p->base[i] = 0;
        p->check[i] = DEAD;
        p->fail[i] = DEAD;
        p->output_pos[i] = 0;
    }
    p->n_slots = n;
}

static int edge_code_cmp(const void *a, const void *b) {
    const edge_t *x = (const edge_t *)a, *y = (const edge_t *)b;
    return x->label < y->label ? -1 : (x->label > y->label ? 1 : 0);
}

/* find_base + verify_base (charwise/builder.rs:320-344); mapped[] = (code, child) by code */
static uint32_t cw_find_base(const orc_pma *p, const helper_t *h, const edge_t *mapped, size_t n) {
    if (h->has_head) {
        uint32_t idx = h->head;
        for (;;) {
            uint32_t base = idx ^ mapped[0].label;
            int ok = 1;
            for (size_t i = 0; ok && i < n; i++)
                if (helper_is_used_index(h, base ^ mapped[i].label)) ok = 0;
            if (ok && base != 0) return base;
            uint32_t next = h->next[helper_off(h, idx)];
            if (next == h->head) break;
            idx = next;
        }
    }
    return (uint32_t)p->n_slots ^ mapped[0].label;
}

static int cw_build_double_array(orc_pma *p, const nfa_t *nfa, uint32_t num_free_blocks) {
    cw_builder b = {p, 0};
    helper_t h;
    /* init_array (charwise/builder.rs:308-318) */
    uint32_t block_len = next_pow2_u32(p->alphabet_size);
    if (block_len < 2) block_len = 2;
    cw_resize(&b, block_len);
    int rc = helper_init(&h, block_len, num_free_blocks);
    if (rc) return rc;
    rc = helper_push_block(&h);
    if (rc) abort();
    helper_use_index(&h, ROOT);
    helper_use_index(&h, DEAD);

    size_t ns = nfa->n_states;
    uint32_t *map = (uint32_t *)xrealloc(NULL, ns * 4);
    for (size_t i = 0; i < ns; i++) map[i] = DEAD;
    map[ROOT] = ROOT;
    uint32_t *stack = (uint32_t *)xrealloc(NULL, (ns + 1) * 4);
    size_t sp = 0;
    stack[sp++] = ROOT;
    edge_t *mapped = NULL;
    size_t cap_mapped = 0;

    /* charwise/builder.rs:251-281 */
    while (sp > 0) {
        uint32_t state_id = stack[--sp];
        const nfa_state *s = &nfa->states[state_id];
        uint32_t state_idx = map[state_id];
        if (s->n_edges == 0) continue;
        if (s->n_edges > cap_mapped) {
            cap_mapped = s->n_edges * 2;
            mapped = (edge_t *)xrealloc(mapped, cap_mapped * sizeof(edge_t));
        }
        const edge_t *e = edges_of(s);
        for (uint32_t i = 0; i < s->n_edges; i++) {
            uint32_t code = mapper_get(p, e[i].label);
            if (code == INVALID_CODE) abort(); /* .unwrap() */
            mapped[i].label = code;
            mapped[i].child = e[i].child;
        }
        qsort(mapped, s->n_edges, sizeof(edge_t), edge_code_cmp); /* sort_unstable_by_key, keys unique */
        uint32_t base = cw_find_base(p, &h, mapped, s->n_edges);
        if (p->n_slots <= (size_t)base) {
            /* extend_array (charwise/builder.rs:346-359) */
            if (p->n_slots > (size_t)(0xffffffffu - block_len)) {
                rc = ORC_AUTOMATON_SCALE;
                goto done;
            }
            rc = helper_push_block(&h);
            if (rc) goto done;
            cw_resize(&b, p->n_slots + block_len);
        }
        for (uint32_t i = 0; i < s->n_edges; i++) {
            uint32_t child_idx = base ^ mapped[i].label;
            helper_use_index(&h, child_idx);
            p->check[child_idx] = state_idx;
            map[mapped[i].child] = child_idx;
            stack[sp++] = mapped[i].child;
        }
        p->base[state_idx] = base;
    }
    /* charwise/builder.rs:284-302 */
    for (size_t i = 0; i < ns; i++) {
        if (i == DEAD) continue;
        uint32_t idx = map[i];
        p->output_pos[idx] = nfa->states[i].output_pos;
        uint32_t fail_id = nfa->states[i].fail;
        p->fail[idx] = fail_id == DEAD ? DEAD : map[fail_id];
    }
    rc = ORC_OK;
done:
    free(map);
    free(stack);
    free(mapped);
    helper_destroy(&h);
    return rc;
}

/* UTF-8 decode as CharWithEndOffsetIterator::next (src/charwise/iter.rs:71-97); unchecked. */
uint32_t orc_utf8_next(const uint8_t *hay, size_t *pos) {
    size_t i = *pos;
    uint32_t first = hay[i++];
    uint32_t c;
    if (first < 0x80) {
        c = first;
    } else {
        uint32_t r = hay[i++] & 0x3f;
        if (first < 0xe0) {
            c = ((first & 0x1f) << 6) | r;
        } else {
            r = (r << 6) | (hay[i++] & 0x3f);
            if (first < 0xf0) {
                c = ((first & 0x0f) << 12) | r;
            } else {
                r = (r << 6) | (hay[i++] & 0x3f);
                c = ((first & 0x07) << 18) | r;
            }
        }
    }
    *pos = i;
    return c;
}

/* build / build_with_values (bytewise/builder.rs:152-244, charwise/builder.rs:129-239) */
int orc_build(int charwise, const uint8_t *bytes, const uint64_t *offs, const uint32_t *values,
              uint32_t n, uint8_t match_kind, uint32_t num_free_blocks, orc_pma **out) {
    *out = NULL;
    if (num_free_blocks == 0) return ORC_INVALID_ARGUMENT; /* assert!(n >= 1) builder.rs:113 */
    if (match_kind > 2) return ORC_INVALID_ARGUMENT;
    nfa_t nfa;
    nfa_init(&nfa, match_kind);
    orc_pma *p = (orc_pma *)calloc(1, sizeof(orc_pma));
    if (!p) abort();
    p->charwise = charwise;
    p->match_kind = match_kind;
    int rc = ORC_OK;
    uint32_t *labels = NULL;
    size_t cap_labels = 0;
    uint32_t *freqs = NULL;
    size_t n_freqs = 0, cap_freqs = 0;

    for (uint32_t i = 0; i < n; i++) {
        const uint8_t *pat = bytes + offs[i];
        size_t plen = (size_t)(offs[i + 1] - offs[i]);
        if (plen + 1 > cap_labels) {
            cap_labels = (plen + 1) * 2;
            labels = (uint32_t *)xrealloc(labels, cap_labels * 4);
        }
        size_t nl = 0;
        if (!charwise) {
            for (size_t k = 0; k < plen; k++) labels[nl++] = pat[k];
        } else {
            size_t pos = 0;
            while (pos < plen) labels[nl++] = orc_utf8_next(pat, &pos); /* .chars() */
        }
        uint32_t value = values ? values[i] : i;
        rc = nfa_add(&nfa, labels, nl, plen, value);
        if (rc) goto fail;
        if (charwise) { /* charwise/builder.rs:222-228 */
            for (size_t k = 0; k < nl; k++) {
                size_t c = labels[k];
                if (n_freqs <= c) {
                    if (c + 1 > cap_freqs) {
                        cap_freqs = (c + 1) * 2;
                        freqs = (uint32_t *)xrealloc(freqs, cap_freqs * 4);
                    }
                    for (size_t z = n_freqs; z < c + 1; z++) freqs[z] = 0;
                    n_freqs = c + 1;
                }
                freqs[c] += 1;
            }
        }
    }
    if (!charwise) {
        if (nfa.len > U24_MAX) { /* bytewise/builder.rs:256-258 */
            rc = ORC_AUTOMATON_SCALE;
            goto fail;
        }
    } else {
        mapper_new(p, freqs, n_freqs);
    }
    {
        size_t qn;
        uint32_t *q = match_kind == ORC_STANDARD ? nfa_build_fails(&nfa, &qn)
                                                 : nfa_build_fails_leftmost(&nfa, &qn);
        nfa_build_outputs(&nfa, q, qn);
        free(q);
    }
    rc = charwise ? cw_build_double_array(p, &nfa, num_free_blocks)
                  : bw_build_double_array(p, &nfa, num_free_blocks);
    if (rc) goto fail;
    if (nfa.n_states - 1 > 0xffffffffull) {
        rc = ORC_AUTOMATON_SCALE;
        goto fail;
    }
    p->num_states = (uint32_t)(nfa.n_states - 1);
    /* shrink to the exact lengths (shrink_to_fit is not observable; lengths are) */
    p->outputs = nfa.outputs;
    p->n_outputs = nfa.n_outputs;
    nfa.outputs = NULL;
    if (!charwise && !is_leftmost(match_kind)) build_root_table(p);
    free(labels);
    free(freqs);
    nfa_destroy(&nfa);
    build_scan_records(p);
    *out = p;
    return ORC_OK;
fail:
    free(labels);
    free(freqs);
    nfa_destroy(&nfa);
    orc_free(p);
    return rc;
}

/* ------------------------------------------------------------------------- */
/* Wire format (src/serializer.rs, src/bytewise.rs:801-964, src/charwise.rs:831-952) */
/* ------------------------------------------------------------------------- */

static void put32(uint8_t **d, uint32_t x) {
    (*d)[0] = (uint8_t)x;
    (*d)[1] = (uint8_t)(x >> 8);
    (*d)[2] = (uint8_t)(x >> 16);
    (*d)[3] = (uint8_t)(x >> 24);
    *d += 4;
}

size_t orc_serialized_bytes(const orc_pma *p) {
    if (!p->charwise) {
        size_t ns = is_leftmost(p->match_kind) ? 0 : p->n_slots;
        size_t nl = is_leftmost(p->match_kind) ? p->n_slots : 0;
        return 4 + ns * 12 + 4 + nl * 8 + 4 + nl * 4 + 4 + p->n_outputs * 12 + 1 + 4;
    }
    return 4 + p->n_slots * 16 + 4 + p->table_len * 4 + 4 + 4 + p->n_outputs * 12 + 1 + 4;
}

size_t orc_serialize(const orc_pma *p, uint8_t *dst, size_t cap) {
    size_t need = orc_serialized_bytes(p);
    if (cap < need) return need;
    uint8_t *d = dst;
    if (!p->charwise) {
        int lm = is_leftmost(p->match_kind);
        /* Vec<State<u32>> */
        put32(&d, lm ? 0 : (uint32_t)p->n_slots);
        if (!lm)
            for (size_t i = 0; i < p->n_slots; i++) {
                put32(&d, p->base[i]);
                put32(&d, p->fail[i]);
                put32(&d, p->opos_ch[i]);
            }
        /* Vec<State<Empty>> */
        put32(&d, lm ? (uint32_t)p->n_slots : 0);
        if (lm)
            for (size_t i = 0; i < p->n_slots; i++) {
                put32(&d, p->base[i]);
                put32(&d, p->opos_ch[i]);
            }
        /* Vec<u32> fails */
        put32(&d, lm ? (uint32_t)p->n_slots : 0);
        if (lm)
            for (size_t i = 0; i < p->n_slots; i++) put32(&d, p->fail[i]);
    } else {
        put32(&d, (uint32_t)p->n_slots);
        for (size_t i = 0; i < p->n_slots; i++) {
            put32(&d, p->base[i]);
            put32(&d, p->check[i]);
            put32(&d, p->fail[i]);
            put32(&d, p->output_pos[i]);
        }
        put32(&d, (uint32_t)p->table_len);
        for (size_t i = 0; i < p->table_len; i++) put32(&d, p->table[i]);
        put32(&d, p->alphabet_size);
    }
    put32(&d, (uint32_t)p->n_outputs);
    for (size_t i = 0; i < p->n_outputs; i++) {
        put32(&d, p->outputs[i].value);
        put32(&d, p->outputs[i].length);
        put32(&d, p->outputs[i].parent);
    }
    *d++ = p->match_kind;
    put32(&d, p->num_states);
    return need;
}

typedef struct {
    const uint8_t *s;
    size_t left;
} rd_t;

static int get32(rd_t *r, uint32_t *x) {
    if (r->left < 4) return 0;
    *x = (uint32_t)r->s[0] | ((uint32_t)r->s[1] << 8) | ((uint32_t)r->s[2] << 16) |
         ((uint32_t)r->s[3] << 24);
    r->s += 4;
    r->left -= 4;
    return 1;
}

/* Vec<S>::deserialize_from_slice header (serializer.rs:112-118): len, then the guard
 * len * size_of::<S>() > remaining => Err. */
static int get_vec_len(rd_t *r, size_t item_bytes, uint32_t *len) {
    if (!get32(r, len)) return 0;
    if ((uint64_t)*len * item_bytes > r->left) return 0;
    return 1;
}

int orc_deserialize(int charwise, const uint8_t *src, size_t len, orc_pma **out, size_t *consumed) {
    *out = NULL;
    rd_t r = {src, len};
    orc_pma *p = (orc_pma *)calloc(1, sizeof(orc_pma));
    if (!p) abort();
    p->charwise = charwise;
    uint32_t n;
#define BAD()                         \
    do {                              \
        orc_free(p);                  \
        return ORC_INVALID_AUTOMATON; \
    } while (0)
    if (!charwise) {
        uint32_t n_states, n_lm, n_fails;
        uint32_t *sb = NULL, *sf = NULL, *so = NULL, *lb = NULL, *lo = NULL, *lf = NULL;
        if (!get_vec_len(&r, 12, &n_states)) BAD();
        sb = (uint32_t *)xrealloc(NULL, (size_t)n_states * 4);
        sf = (uint32_t *)xrealloc(NULL, (size_t)n_states * 4);
        so = (uint32_t *)xrealloc(NULL, (size_t)n_states * 4);
        p->base = sb;
        p->fail = sf;
        p->opos_ch = so;
        for (uint32_t i = 0; i < n_states; i++)
            if (!get32(&r, &sb[i]) || !get32(&r, &sf[i]) || !get32(&r, &so[i])) BAD();
        if (!get_vec_len(&r, 8, &n_lm)) BAD();
        lb = (uint32_t *)xrealloc(NULL, (size_t)n_lm * 4);
        lo = (uint32_t *)xrealloc(NULL, (size_t)n_lm * 4);
        for (uint32_t i = 0; i < n_lm; i++)
            if (!get32(&r, &lb[i]) || !get32(&r, &lo[i])) {
                free(lb);
                free(lo);
                BAD();
            }
        if (!get_vec_len(&r, 4, &n_fails)) {
            free(lb);
            free(lo);
            BAD();
        }
        lf = (uint32_t *)xrealloc(NULL, (size_t)n_fails * 4);
        for (uint32_t i = 0; i < n_fails; i++)
            if (!get32(&r, &lf[i])) {
                free(lb);
                free(lo);
                free(lf);
                BAD();
            }
#define BADL()    \
    do {          \
        free(lb); \
        free(lo); \
        free(lf); \
        BAD();    \
    } while (0)
        if (!get_vec_len(&r, 12, &n)) BADL();
        p->outputs = (output_t *)xrealloc(NULL, (size_t)n * sizeof(output_t));
        p->n_outputs = n;
        for (uint32_t i = 0; i < n; i++)
            if (!get32(&r, &p->outputs[i].value) || !get32(&r, &p->outputs[i].length) ||
                !get32(&r, &p->outputs[i].parent))
                BADL();
        if (r.left < 1) BADL();
        uint8_t mk = r.s[0];
        r.s++;
        r.left--;
        p->match_kind = (mk == 1 || mk == 2) ? mk : 0; /* From<u8> (src/lib.rs:362-370) */
        if (!get32(&r, &p->num_states)) BADL();
        /* validation (src/bytewise.rs:892-962) */
        if (is_leftmost(p->match_kind)) {
            if (n_states != 0) BADL();
            if (n_lm == 0) BADL();
            if (n_lm % 256 != 0) BADL();
            if (n_fails != n_lm) BADL();
            for (uint32_t i = 0; i < n_lm; i++) {
                if (lb[i] != 0 && lb[i] >= n_lm) BADL();
                uint32_t op = lo[i] >> 8;
                if (op != 0 && op - 1 >= p->n_outputs) BADL();
            }
            for (uint32_t i = 0; i < n_fails; i++)
                if (lf[i] >= n_lm) BADL();
            free(sb);
            free(sf);
            free(so);
            p->base = lb;
            p->opos_ch = lo;
            p->fail = lf;
            p->n_slots = n_lm;
        } else {
            if (n_lm != 0 || n_fails != 0) BADL();
            if (n_states == 0) BADL();
            if (n_states % 256 != 0) BADL();
            for (uint32_t i = 0; i < n_states; i++) {
                if (sb[i] != 0 && sb[i] >= n_states) BADL();
                if (sf[i] >= n_states) BADL();
                uint32_t op = so[i] >> 8;
                if (op != 0 && op - 1 >= p->n_outputs) BADL();
            }
            free(lb);
            free(lo);
            free(lf);
            p->n_slots = n_states;
            build_root_table(p);
        }
    } else {
        if (!get_vec_len(&r, 16, &n)) BAD();
        p->n_slots = n;
        p->base = (uint32_t *)xrealloc(NULL, (size_t)n * 4);
        p->check = (uint32_t *)xrealloc(NULL, (size_t)n * 4);
        p->fail = (uint32_t *)xrealloc(NULL, (size_t)n * 4);
        p->output_pos = (uint32_t *)xrealloc(NULL, (size_t)n * 4);
        for (uint32_t i = 0; i < n; i++)
            if (!get32(&r, &p->base[i]) || !get32(&r, &p->check[i]) || !get32(&r, &p->fail[i]) ||
                !get32(&r, &p->output_pos[i]))
                BAD();
        if (!get_vec_len(&r, 4, &n)) BAD();
        p->table_len = n;
        p->table = (uint32_t *)xrealloc(NULL, (size_t)n * 4);
        for (uint32_t i = 0; i < n; i++)
            if (!get32(&r, &p->table[i])) BAD();
        if (!get32(&r, &p->alphabet_size)) BAD();
        if (!get_vec_len(&r, 12, &n)) BAD();
        p->outputs = (output_t *)xrealloc(NULL, (size_t)n * sizeof(output_t));
        p->n_outputs = n;
        for (uint32_t i = 0; i < n; i++)
            if (!get32(&r, &p->outputs[i].value) || !get32(&r, &p->outputs[i].length) ||
                !get32(&r, &p->outputs[i].parent))
                BAD();
        if (r.left < 1) BAD();
        uint8_t mk = r.s[0];
        r.s++;
        r.left--;
        p->match_kind = (mk == 1 || mk == 2) ? mk : 0;
        if (!get32(&r, &p->num_states)) BAD();
        /* validation (src/charwise.rs:912-943) */
        for (size_t i = 0; i < p->table_len; i++) {
            if (p->table[i] == INVALID_CODE) continue;
            if (p->table[i] >= p->alphabet_size) BAD();
        }
        size_t block_len = next_pow2_u32(p->alphabet_size);
        if (block_len < 2) block_len = 2;
        if (p->n_slots == 0) BAD();
        if (p->n_slots % block_len != 0) BAD();
        for (size_t i = 0; i < p->n_slots; i++) {
            if (p->base[i] != 0 && p->base[i] >= p->n_slots) BAD();
            if (p->fail[i] >= p->n_slots) BAD();
            if (p->output_pos[i] != 0 && p->output_pos[i] - 1 >= p->n_outputs) BAD();
        }
    }
    /* src/bytewise.rs:956-962, src/charwise.rs:944-950 */
    for (size_t i = 0; i < p->n_outputs; i++) {
        uint32_t parent = p->outputs[i].parent;
        if (parent != 0 && (size_t)(parent - 1) >= i) BAD();
    }
#undef BADL
#undef BAD
    if (consumed) *consumed = len - r.left;
    build_scan_records(p);
    *out = p;
    return ORC_OK;
}

/* ------------------------------------------------------------------------- */
/* Introspection                                                               */
/* ------------------------------------------------------------------------- */

int orc_is_charwise(const orc_pma *p) { return p->charwise; }
uint8_t orc_match_kind(const orc_pma *p) { return p->match_kind; }
uint32_t orc_num_states(const orc_pma *p) { return p->num_states; }
size_t orc_num_elements(const orc_pma *p) { return p->n_slots; }
size_t orc_num_outputs(const orc_pma *p) { return p->n_outputs; }
uint32_t orc_alphabet_size(const orc_pma *p) { return p->alphabet_size; }

/* heap_bytes (src/bytewise.rs:764-770, src/charwise.rs:813-817) */
size_t orc_heap_bytes(const orc_pma *p) {
    if (!p->charwise) {
        if (is_leftmost(p->match_kind)) return p->n_slots * 8 + p->n_slots * 4 + p->n_outputs * 12;
        return p->n_slots * 12 + 256 * 4 + p->n_outputs * 12;
    }
    return p->n_slots * 16 + p->table_len * 4 + p->n_outputs * 12;
}

uint32_t orc_max_pattern_len(const orc_pma *p) {
    uint32_t m = 0;
    for (size_t i = 0; i < p->n_outputs; i++)
        if (p->outputs[i].length > m) m = p->outputs[i].length;
    return m;
}

int orc_peek_state(const orc_pma *p, size_t idx, uint32_t *base, uint32_t *check, uint32_t *fail,
                   uint32_t *output_pos) {
    if (idx >= p->n_slots) return 1;
    *base = p->base[idx];
    *fail = p->fail[idx];
    if (!p->charwise) {
        *check = p->opos_ch[idx] & 0xff;
        *output_pos = p->opos_ch[idx] >> 8;
    } else {
        *check = p->check[idx];
        *output_pos = p->output_pos[idx];
    }
    return 0;
}

uint32_t orc_mapper_get(const orc_pma *p, uint32_t c) { return mapper_get(p, c); }

/* ------------------------------------------------------------------------- */
/* Transitions                                                                 */
/* ------------------------------------------------------------------------- */

/* next_state_id_unchecked (src/bytewise.rs:1063-1088) */
static inline uint32_t bw_next(const orc_pma *p, uint32_t s, uint32_t c) {
    const struct bw_state *st = p->st12;
    for (;;) {
        if (s == ROOT) return p->root_table[c];
        uint32_t b = st[s].base;
        if (b != 0) {
            uint32_t child = b ^ c;
            if ((st[child].opos_ch & 0xff) == c) return child;
        }
        s = st[s].fail;
    }
}

/* next_state_id_leftmost_unchecked (src/bytewise.rs:1094-1128) */
static inline uint32_t bw_next_leftmost(const orc_pma *p, uint32_t s, uint32_t c) {
    const struct lm_state *st = p->st8;
    for (;;) {
        uint32_t b = st[s].base;
        if (b != 0) {
            uint32_t child = b ^ c;
            if ((st[child].opos_ch & 0xff) == c) return child;
        }
        if (s == ROOT) return ROOT;
        uint32_t f = p->fail[s];
        if (f == DEAD) return ROOT;
        s = f;
    }
}

/* next_state_id_unchecked (src/charwise.rs:1022-1051) */
static inline uint32_t cw_next(const orc_pma *p, uint32_t s, uint32_t cp) {
    uint32_t mc = mapper_get(p, cp);
    if (mc == INVALID_CODE) return ROOT;
    const struct cw_state *st = p->st16;
    for (;;) {
        uint32_t b = st[s].base;
        if (b != 0) {
            uint32_t child = b ^ mc;
            if (st[child].check == s) return child;
        }
        if (s == ROOT) return ROOT;
        s = st[s].fail;
    }
}

/* next_state_id_leftmost_unchecked (src/charwise.rs:1057-1092) */
static inline uint32_t cw_next_leftmost(const orc_pma *p, uint32_t s, uint32_t cp) {
    uint32_t mc = mapper_get(p, cp);
    if (mc == INVALID_CODE) return ROOT;
    const struct cw_state *st = p->st16;
    for (;;) {
        uint32_t b = st[s].base;
        if (b != 0) {
            uint32_t child = b ^ mc;
            if (st[child].check == s) return child;
        }
        if (s == ROOT) return ROOT;
        uint32_t f = st[s].fail;
        if (f == DEAD) return ROOT;
        s = f;
    }
}

static inline uint32_t st_opos(const orc_pma *p, uint32_t s) {
    if (p->st12) return p->st12[s].opos_ch >> 8;
    if (p->st16) return p->st16[s].output_pos;
    return p->st8[s].opos_ch >> 8;
}

/* ------------------------------------------------------------------------- */
/* Scans                                                                       */
/* ------------------------------------------------------------------------- */

uint64_t orc_hash_step(uint64_t h, uint32_t start, uint32_t end, uint32_t value) {
    /* order-sensitive: FNV-style fold of the three words, then a multiply-xorshift */
    h ^= (uint64_t)start + 0x9e3779b97f4a7c15ull;
    h *= 0x100000001b3ull;
    h ^= (uint64_t)end + 0xc2b2ae3d27d4eb4full;
    h *= 0x100000001b3ull;
    h ^= (uint64_t)value + 0x165667b19e3779f9ull;
    h *= 0x100000001b3ull;
    h ^= h >> 29;
    return h;
}

/* per-haystack order-sensitive hashes of an existing result (matches + n+1 offsets): what orc_scan_batch
 * reports in `hashes`, computed from another implementation's output so that the two can be compared
 * without moving the tuples around */
void orc_hash_matches(const orc_match *m, const uint64_t *offs, uint64_t n, uint64_t *hashes) {
    for (uint64_t i = 0; i < n; i++) {
        uint64_t h = 0;
        for (uint64_t k = offs[i]; k < offs[i + 1]; k++) h = orc_hash_step(h, m[k].start, m[k].end, m[k].value);
        hashes[i] = h;
    }
}

typedef struct {
    orc_match *out;
    size_t cap, n;
    uint64_t hash;
    int want_hash;   /* 0: the timed baseline does not pay for the checker's hash */
    orc_match *ring; /* timed baseline: every match is stored like a consumer collecting them would, into a
                        small per-thread ring (ring_mask + 1 entries) instead of an unbounded Vec */
    size_t ring_mask;
} sink_t;

static inline void emit(sink_t *k, size_t end, uint32_t length, uint32_t value) {
    uint32_t st = (uint32_t)(end - length), en = (uint32_t)end;
    if (k->out && k->n < k->cap) {
        k->out[k->n].start = st;
        k->out[k->n].end = en;
        k->out[k->n].value = value;
    }
    if (k->ring) {
        orc_match *m = &k->ring[k->n & k->ring_mask];
        m->start = st;
        m->end = en;
        m->value = value;
    }
    if (k->want_hash) k->hash = orc_hash_step(k->hash, st, en, value);
    k->n++;
}

/* FindOverlappingIterator (bytewise/iter.rs:133-176; charwise/iter.rs:190-235) */
static void scan_overlapping(const orc_pma *p, const uint8_t *hay, size_t len, sink_t *k) {
    uint32_t s = ROOT;
    /* the iterator starts with output_pos = ROOT's (src/bytewise.rs:307-311), pos = 0 */
    for (uint32_t op = st_opos(p, ROOT); op != 0; op = p->outputs[op - 1].parent)
        emit(k, 0, p->outputs[op - 1].length, p->outputs[op - 1].value);
    size_t i = 0;
    while (i < len) {
        size_t end;
        if (!p->charwise) {
            s = bw_next(p, s, hay[i]);
            end = ++i;
        } else {
            uint32_t cp = orc_utf8_next(hay, &i);
            end = i;
            s = cw_next(p, s, cp);
        }
        for (uint32_t op = st_opos(p, s); op != 0; op = p->outputs[op - 1].parent)
            emit(k, end, p->outputs[op - 1].length, p->outputs[op - 1].value);
    }
}

/* FindOverlappingNoSuffixIterator (bytewise/iter.rs:195-243; charwise/iter.rs:254-302) */
static void scan_overlapping_no_suffix(const orc_pma *p, const uint8_t *hay, size_t len, sink_t *k) {
    uint32_t s = ROOT;
    uint32_t rop = st_opos(p, ROOT);
    if (rop != 0) emit(k, 0, 0, p->outputs[rop - 1].value); /* first_call: length 0, end 0 */
    size_t i = 0;
    while (i < len) {
        size_t end;
        if (!p->charwise) {
            s = bw_next(p, s, hay[i]);
            end = ++i;
        } else {
            uint32_t cp = orc_utf8_next(hay, &i);
            end = i;
            s = cw_next(p, s, cp);
        }
        uint32_t op = st_opos(p, s);
        if (op != 0) emit(k, end, p->outputs[op - 1].length, p->outputs[op - 1].value);
    }
}

/* FindIterator (bytewise/iter.rs:58-113; charwise/iter.rs:115-170) */
static void scan_find(const orc_pma *p, const uint8_t *hay, size_t len, sink_t *k) {
    uint32_t rop = st_opos(p, ROOT);
    size_t i = 0;
    if (rop != 0) {
        /* an empty pattern exists: only zero-length matches, one per boundary */
        uint32_t v = p->outputs[rop - 1].value;
        emit(k, 0, 0, v);
        while (i < len) {
            if (!p->charwise)
                i++;
            else
                (void)orc_utf8_next(hay, &i);
            emit(k, i, 0, v);
        }
        return;
    }
    while (i < len) {
        uint32_t s = ROOT; /* every next() restarts from ROOT (iter.rs:87) */
        int found = 0;
        while (i < len) {
            size_t end;
            if (!p->charwise) {
                s = bw_next(p, s, hay[i]);
                end = ++i;
            } else {
                uint32_t cp = orc_utf8_next(hay, &i);
                end = i;
                s = cw_next(p, s, cp);
            }
            uint32_t op = st_opos(p, s);
            if (op != 0) {
                emit(k, end, p->outputs[op - 1].length, p->outputs[op - 1].value);
                found = 1;
                break;
            }
        }
        if (!found) break;
    }
}

/* LeftmostFindIterator (bytewise/iter.rs:272-340; charwise/iter.rs:328-399).  The state
 * of the iterator (pos, init_output_pos, skip_empty) lives across next() calls; each
 * turn of the outer for(;;) below is one next() call. */
static void scan_leftmost(const orc_pma *p, const uint8_t *hay, size_t len, sink_t *k) {
    size_t self_pos = 0;
    uint32_t init_output_pos = st_opos(p, ROOT);
    int skip_empty = 0;
    for (;;) { /* one next() */
        uint32_t s = ROOT;
        uint32_t last = init_output_pos;
        int yielded = 0;
    restart: /* 'a: loop */
    {
        size_t i = self_pos;
        while (i < len) {
            size_t unit_start = i, unit_end;
            if (!p->charwise) {
                s = bw_next_leftmost(p, s, hay[i]);
                unit_end = ++i;
            } else {
                uint32_t cp = orc_utf8_next(hay, &i);
                unit_end = i;
                s = cw_next_leftmost(p, s, cp);
            }
            (void)unit_start;
            if (s == ROOT) {
                if (last != 0) {
                    size_t end = self_pos;
                    if (last == init_output_pos) {
                        /* bytewise: self.pos += 1; charwise: self.pos += c.len_utf8() */
                        self_pos += unit_end - unit_start;
                        /* DOCUMENTED DIVERGENCE (DESIGN.md "Reference divergences"): c is the char that
                         * fell back to ROOT, not the char at self.pos, so with chars of mixed byte
                         * lengths self.pos can land inside a char; the reference then slices the &str
                         * off a char boundary (charwise/iter.rs:334, undefined behaviour).  We move on
                         * to the next char boundary (at most 3 continuation bytes). */
                        if (p->charwise) {
                            int k = 0;
                            while (k < 3 && self_pos < len && (hay[self_pos] & 0xC0) == 0x80) ++self_pos, ++k;
                        }
                        if (skip_empty) {
                            skip_empty = 0;
                            goto restart;
                        }
                    } else {
                        skip_empty = 1;
                    }
                    emit(k, end, p->outputs[last - 1].length, p->outputs[last - 1].value);
                    yielded = 1;
                    break;
                }
            } else {
                uint32_t op = st_opos(p, s);
                if (op != 0) {
                    last = op;
                    self_pos = unit_end; /* pos + 1  /  self.pos += skips */
                }
            }
        }
    }
        if (yielded) continue;
        /* after the loop (iter.rs:320-339) */
        if (self_pos >= len) init_output_pos = 0; /* > only on invalid UTF-8 (a char cut off by the end) */
        if (last != 0) {
            if (self_pos < len && last == init_output_pos) {
                /* DOCUMENTED DIVERGENCE (DESIGN.md "Reference divergences"): the input ended inside
                 * a partial match while only the empty pattern is pending.  The reference returns
                 * this empty match WITHOUT advancing self.pos (iter.rs:320-335), so its iterator
                 * never terminates on such input.  We treat end-of-input like the fall-back-to-ROOT
                 * branch (iter.rs:283-293): consume one unit at self.pos, honour skip_empty. */
                size_t end = self_pos;
                if (!p->charwise) {
                    self_pos += 1;
                } else {
                    size_t t = self_pos;
                    (void)orc_utf8_next(hay, &t);
                    self_pos = t;
                }
                if (skip_empty) {
                    skip_empty = 0;
                    continue;
                }
                emit(k, end, p->outputs[last - 1].length, p->outputs[last - 1].value);
                continue;
            }
            emit(k, self_pos, p->outputs[last - 1].length, p->outputs[last - 1].value);
            continue;
        }
        self_pos = len;
        return; /* None */
    }
}

/* FindStepper driven byte by byte / char by char, collecting matches() after every
 * consume() and once before (tests/aho_corasick_crate_test.rs:422-463;
 * bytewise/iter.rs:357-400, charwise/iter.rs:416-459). */
static void scan_find_stepper(const orc_pma *p, const uint8_t *hay, size_t len, sink_t *k) {
    uint32_t s = ROOT;
    size_t pos = 0;
    uint32_t output_pos = st_opos(p, ROOT);
    if (output_pos != 0) emit(k, pos, p->outputs[output_pos - 1].length, p->outputs[output_pos - 1].value);
    size_t i = 0;
    while (i < len) {
        uint32_t unit;
        if (!p->charwise) {
            unit = hay[i++];
        } else {
            unit = orc_utf8_next(hay, &i);
        }
        pos = i;
        if (st_opos(p, ROOT) == 0) {
            s = p->charwise ? cw_next(p, s, unit) : bw_next(p, s, unit);
            output_pos = st_opos(p, s);
            if (output_pos != 0) s = ROOT;
        }
        if (output_pos != 0)
            emit(k, pos, p->outputs[output_pos - 1].length, p->outputs[output_pos - 1].value);
    }
}

/* FindOverlappingStepper (bytewise/iter.rs:450-474; tests :477-520) */
static void scan_overlapping_stepper(const orc_pma *p, const uint8_t *hay, size_t len, sink_t *k) {
    uint32_t s = ROOT;
    for (uint32_t op = st_opos(p, s); op != 0; op = p->outputs[op - 1].parent)
        emit(k, 0, p->outputs[op - 1].length, p->outputs[op - 1].value);
    size_t i = 0;
    while (i < len) {
        if (!p->charwise) {
            s = bw_next(p, s, hay[i++]);
        } else {
            uint32_t cp = orc_utf8_next(hay, &i);
            s = cw_next(p, s, cp);
        }
        for (uint32_t op = st_opos(p, s); op != 0; op = p->outputs[op - 1].parent)
            emit(k, i, p->outputs[op - 1].length, p->outputs[op - 1].value);
    }
}

static int mode_ok(const orc_pma *p, int mode) {
    /* asserts of src/bytewise.rs:194-197, 299-302, 551-554 and charwise twins */
    if (mode == ORC_LEFTMOST_FIND) return is_leftmost(p->match_kind);
    return !is_leftmost(p->match_kind);
}

static void scan_one(const orc_pma *p, int mode, const uint8_t *hay, size_t len, sink_t *k) {
    switch (mode) {
        case ORC_FIND: scan_find(p, hay, len, k); break;
        case ORC_FIND_OVERLAPPING: scan_overlapping(p, hay, len, k); break;
        case ORC_FIND_OVERLAPPING_NO_SUFFIX: scan_overlapping_no_suffix(p, hay, len, k); break;
        case ORC_LEFTMOST_FIND: scan_leftmost(p, hay, len, k); break;
        case ORC_FIND_STEPPER: scan_find_stepper(p, hay, len, k); break;
        case ORC_FIND_OVERLAPPING_STEPPER: scan_overlapping_stepper(p, hay, len, k); break;
        default: break;
    }
}

int orc_scan(const orc_pma *p, int mode, const uint8_t *hay, size_t len, orc_match *out, size_t cap,
             size_t *n_out) {
    if (mode < 0 || mode > ORC_FIND_OVERLAPPING_STEPPER) return ORC_INVALID_ARGUMENT;
    if (!mode_ok(p, mode)) return ORC_MATCH_KIND_MISMATCH;
    sink_t k = {out, cap, 0, 0, 1, NULL, 0};
    scan_one(p, mode, hay, len, &k);
    if (n_out) *n_out = k.n;
    return ORC_OK;
}

/* ---- batch ---------------------------------------------------------------- */

typedef struct {
    const orc_pma *p;
    int mode;
    const uint8_t *text;
    const uint64_t *offs;
    uint64_t n;
    uint64_t *counts, *hashes;
    orc_match *out;
    const uint64_t *out_offs; /* pass 2: per-haystack start in out */
    uint64_t out_cap;
    int store_ring; /* timed baseline: matches go to a per-thread ring */
} job_t;

/* A persistent pool of worker threads, each pinned to one of the CPUs this process may run on (the crate's
 * users would use rayon or std::thread the same way); haystacks are handed out in chunks from one atomic
 * counter.  The pool is (re)built when the requested thread count changes. */
#define POOL_CHUNK 16
#define RING_ENTRIES 4096
typedef struct {
    pthread_t th;
    int index;
    orc_match *ring;
} worker_t;
static struct {
    pthread_mutex_t mu;
    pthread_cond_t go, done;
    worker_t *w;
    int n_workers, running, generation, quit;
    job_t job;
    volatile uint64_t next;
} g_pool = {PTHREAD_MUTEX_INITIALIZER, PTHREAD_COND_INITIALIZER, PTHREAD_COND_INITIALIZER, NULL, 0, 0, 0, 0, {0}, 0};

static void run_chunk(const job_t *j, uint64_t lo, uint64_t hi, orc_match *ring) {
    for (uint64_t i = lo; i < hi; i++) {
        const uint8_t *hay = j->text + j->offs[i];
        size_t len = (size_t)(j->offs[i + 1] - j->offs[i]);
        sink_t k = {NULL, 0, 0, 0, j->hashes != NULL, NULL, 0};
        if (j->out_offs) {
            uint64_t o = j->out_offs[i];
            k.out = j->out + o;
            k.cap = o < j->out_cap ? (size_t)(j->out_cap - o) : 0;
        } else if (j->store_ring) {
            k.ring = ring;
            k.ring_mask = RING_ENTRIES - 1;
        }
        scan_one(j->p, j->mode, hay, len, &k);
        if (!j->out_offs) {
            j->counts[i] = k.n;
            if (j->hashes) j->hashes[i] = k.hash;
        }
    }
}

static void drain_items(const job_t *j, orc_match *ring) {
    for (;;) {
        const uint64_t lo = __atomic_fetch_add(&g_pool.next, POOL_CHUNK, __ATOMIC_RELAXED);
        if (lo >= j->n) break;
        run_chunk(j, lo, lo + POOL_CHUNK < j->n ? lo + POOL_CHUNK : j->n, ring);
    }
}

static void *pool_worker(void *arg) {
    worker_t *w = (worker_t *)arg;
    int seen = 0;
    pthread_mutex_lock(&g_pool.mu);
    for (;;) {
        while (!g_pool.quit && g_pool.generation == seen) pthread_cond_wait(&g_pool.go, &g_pool.mu);
        if (g_pool.quit) break;
        seen = g_pool.generation;
        pthread_mutex_unlock(&g_pool.mu);
        drain_items(&g_pool.job, w->ring);
        pthread_mutex_lock(&g_pool.mu);
        if (--g_pool.running == 0) pthread_cond_signal(&g_pool.done);
    }
    pthread_mutex_unlock(&g_pool.mu);
    return NULL;
}

static void pool_stop(void) {
    if (!g_pool.w) return;
    pthread_mutex_lock(&g_pool.mu);
    g_pool.quit = 1;
    pthread_cond_broadcast(&g_pool.go);
    pthread_mutex_unlock(&g_pool.mu);
    for (int t = 0; t < g_pool.n_workers; t++) {
        pthread_join(g_pool.w[t].th, NULL);
        free(g_pool.w[t].ring);
    }
    free(g_pool.w);
    g_pool.w = NULL;
    g_pool.n_workers = 0;
    g_pool.quit = 0;
}

static void pool_start(int nthreads) {
    cpu_set_t allowed;
    int cpus[1024], n_cpus = 0;
    if (sched_getaffinity(0, sizeof(allowed), &allowed) == 0)
        for (int c = 0; c < 1024 && c < CPU_SETSIZE; c++)
            if (CPU_ISSET(c, &allowed)) cpus[n_cpus++] = c;
    g_pool.w = (worker_t *)xrealloc(NULL, sizeof(worker_t) * (size_t)nthreads);
    g_pool.n_workers = nthreads;
    for (int t = 0; t < nthreads; t++) {
        g_pool.w[t].index = t;
        g_pool.w[t].ring = (orc_match *)xrealloc(NULL, sizeof(orc_match) * RING_ENTRIES);
        if (pthread_create(&g_pool.w[t].th, NULL, pool_worker, &g_pool.w[t]) != 0) abort();
        if (n_cpus > 0) {
            cpu_set_t one;
            CPU_ZERO(&one);
            CPU_SET(cpus[t % n_cpus], &one);
            pthread_setaffinity_np(g_pool.w[t].th, sizeof(one), &one);
        }
    }
}

static void run_jobs(job_t *proto, uint64_t n, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    proto->n = n;
    if (nthreads == 1 || n <= POOL_CHUNK) {
        orc_match *ring = proto->store_ring ? (orc_match *)xrealloc(NULL, sizeof(orc_match) * RING_ENTRIES) : NULL;
        run_chunk(proto, 0, n, ring);
        free(ring);
        return;
    }
    static pthread_mutex_t serial = PTHREAD_MUTEX_INITIALIZER; /* one batch at a time owns the pool */
    pthread_mutex_lock(&serial);
    if (g_pool.n_workers != nthreads) {
        pool_stop();
        pool_start(nthreads);
    }
    pthread_mutex_lock(&g_pool.mu);
    g_pool.job = *proto;
    g_pool.next = 0;
    g_pool.running = g_pool.n_workers;
    g_pool.generation++;
    pthread_cond_broadcast(&g_pool.go);
    while (g_pool.running) pthread_cond_wait(&g_pool.done, &g_pool.mu);
    pthread_mutex_unlock(&g_pool.mu);
    pthread_mutex_unlock(&serial);
}

/* The timed CPU baseline (bench.py cpu_baseline / --impl reference): the scan loops above on the crate's
 * record layout, persistent pinned threads, every match stored into a per-thread ring, no checker hash.
 * Returns the total match count in *total. */
int orc_bench_batch(const orc_pma *p, int mode, const uint8_t *text, const uint64_t *offs, uint64_t n, int nthreads,
                    uint64_t *counts, uint64_t *total) {
    if (mode < 0 || mode > ORC_FIND_OVERLAPPING_STEPPER) return ORC_INVALID_ARGUMENT;
    if (!mode_ok(p, mode)) return ORC_MATCH_KIND_MISMATCH;
    uint64_t *own = NULL;
    if (!counts) counts = own = (uint64_t *)xrealloc(NULL, (n ? n : 1) * 8);
    job_t proto;
    memset(&proto, 0, sizeof(proto));
    proto.p = p;
    proto.mode = mode;
    proto.text = text;
    proto.offs = offs;
    proto.counts = counts;
    proto.store_ring = 1;
    run_jobs(&proto, n, nthreads);
    uint64_t tot = 0;
    for (uint64_t i = 0; i < n; i++) tot += counts[i];
    if (total) *total = tot;
    free(own);
    return ORC_OK;
}

int orc_scan_batch(const orc_pma *p, int mode, const uint8_t *text, const uint64_t *offs, uint64_t n,
                   int nthreads, uint64_t *counts, uint64_t *hashes, orc_match *out, uint64_t out_cap,
                   uint64_t *total) {
    if (mode < 0 || mode > ORC_FIND_OVERLAPPING_STEPPER) return ORC_INVALID_ARGUMENT;
    if (!mode_ok(p, mode)) return ORC_MATCH_KIND_MISMATCH;
    uint64_t *own_counts = NULL;
    if (!counts) counts = own_counts = (uint64_t *)xrealloc(NULL, (n ? n : 1) * 8);
    job_t proto;
    memset(&proto, 0, sizeof(proto));
    proto.p = p;
    proto.mode = mode;
    proto.text = text;
    proto.offs = offs;
    proto.counts = counts;
    proto.hashes = hashes;
    run_jobs(&proto, n, nthreads);
    uint64_t tot = 0;
    for (uint64_t i = 0; i < n; i++) tot += counts[i];
    if (total) *total = tot;
    if (out) {
        uint64_t *oo = (uint64_t *)xrealloc(NULL, (n + 1) * 8);
        uint64_t acc = 0;
        for (uint64_t i = 0; i < n; i++) {
            oo[i] = acc;
            acc += counts[i];
        }
        oo[n] = acc;
        proto.out = out;
        proto.out_offs = oo;
        proto.out_cap = out_cap;
        run_jobs(&proto, n, nthreads);
        free(oo);
    }
    free(own_counts);
    return ORC_OK;
}
