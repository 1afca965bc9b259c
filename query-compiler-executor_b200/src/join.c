/* join.c -- join operator on the GPU.
 *
 * Same contract as execute_join, /root/reference/src/join.c:630-679.  The
 * host keeps the part that is tiny, serial and decides what runs -- the
 * mid-result state machine -- and every loop over tuples is a kernel behind
 * the C-ABI (include/qce_b200.h):
 *
 *   reference (src/join.c)                      here
 *   build_relations :152-292                    plan_join()      host, O(#entries)
 *   allocate_relation(_mid_results) :96-142     qce_build_tuples_base / _rowids
 *   iterative_sort :5-94                        qce_sort_tuples
 *   join_relations :325-392                     qce_merge_join
 *   scan_join :395-423                          qce_scan_join / qce_scan_join_base
 *   Hashmap dedup :358-367                      qce_distinct_pairs, only when a
 *                                               bystander column needs it
 *   join_payloads :426-484                      qce_rejoin
 *   update_mid_results / fix_all :486-628       install_results()  host
 *
 * The state machine is mirrored decision for decision (including the
 * asymmetric constants of :253-267 and the relation-id bystander test of
 * :495), because it selects which kernels run and so defines the reference's
 * output.  A JOIN_SORT_RHS merge whose "already sorted" lhs is in fact not
 * sorted is computed with the closed form of the reference's pointer walk
 * (qce_merge_join_walk).  One case is refused with a diagnostic: a JOIN_SORT_LHS
 * merge whose *inner* (rhs) run is not sorted -- the walk's result there is a
 * serial scan over an unsorted array (SURVEY.md 8a-10), outside the
 * parity-defined query class.
 */
#include "join.h"

#include "../../include/qce_b200.h"
#include "schedule.h"

/* ---- bystander re-join elision (SURVEY.md 8f-2) ------------------------------------------------
 * join_payloads (src/join.c:426-484) re-aligns every other column of an entity after a join with
 * a distinct-pair pass, two sorts and a merge PER COLUMN.  Inside the parity-defined query class
 * the multiset it produces is {B[i] x matches(U[i])} -- exactly what gathering B through the
 * POSITIONS of the joined column's tuples gives (qce_build_tuples_positions + qce_rowids_gather).
 * The two differ only in the ORDER of the re-joined column (the reference's is by row id of U,
 * the gathered one stays aligned with U'), which the reference itself never relies on inside the
 * class: it matters only when a later operator pairs columns of that entity positionally, and
 * then the reference's own result is pairing-dependent unless every tuple has the same number of
 * matches.  So a query runs in elided mode while, per join with bystanders,
 *   - the other side is a base relation (distinct row ids: matches == distinct partners),
 *   - the entity has not been re-joined before, OR every outer tuple has the same match count
 *     (min == max, qce_merge_join_stats) -- then any pairing yields the same multiset,
 * and no positional operator (scan_join, a JOIN_SORT_* that trusts an order, a refine) touches an
 * entity that has been re-joined.  Anything else raises `unsafe`: the scheduler discards the
 * attempt and replays the query faithfully (schedule.c), so nothing is ever answered differently. */
#define MAX_TRACKED_ENTITIES 16
static __thread int tl_elide = 0, tl_unsafe = 0;
static __thread DArray *tl_rejoined[MAX_TRACKED_ENTITIES];
static __thread int tl_nrejoined = 0;

void qce_join_elide_begin(int on)
{
    tl_elide = on;
    tl_unsafe = 0;
    tl_nrejoined = 0;
}
int qce_join_elide_unsafe(void) { return tl_unsafe; }
int qce_join_elide_active(void) { return tl_elide && !tl_unsafe; }
void qce_join_elide_raise(void) { tl_unsafe = 1; }

static int entity_rejoined(const DArray *entity)
{
    for (int i = 0; i < tl_nrejoined; i++)
        if (tl_rejoined[i] == entity) return 1;
    return 0;
}
static void mark_rejoined(DArray *entity)
{
    if (entity_rejoined(entity)) return;
    if (tl_nrejoined == MAX_TRACKED_ENTITIES) { tl_unsafe = 1; return; }
    tl_rejoined[tl_nrejoined++] = entity;
}
int qce_entity_was_rejoined(const DArray *entity) { return entity_rejoined(entity); }

/* one operand of the predicate, resolved against the entity list */
typedef struct join_side {
    uint32_t rel;       /* relation id */
    uint64_t binding;   /* binding index in the query */
    uint32_t col;       /* join column */
    mid_result *source; /* row-id column the tuples are built from; NULL = base column */
} join_side;

typedef struct join_plan {
    int kind;
    join_side lhs, rhs;
} join_plan;

static mid_result *entry_at(DArray *entities, exists_info where)
{
    DArray *entity = *(DArray **)DArray_get(entities, where.mid_result);
    return (mid_result *)DArray_get(entity, where.index);
}

static DArray *push_entity(DArray *entities)
{
    DArray *fresh = DArray_create(sizeof(mid_result), 4);
    if (fresh != NULL) DArray_push(entities, &fresh);
    return fresh;
}

/* Decide the join kind and where each side's tuples come from.
 * Decision table of build_relations, src/join.c:152-292:
 *   (0) same relation id and same column (bindings ignored)        -> DO_NOTHING
 *   (1) lhs in the current (last) entity, rhs not                  -> :181-220
 *   (2) both in the current entity                                 -> SCAN_JOIN
 *   (3) rhs in the current entity, lhs not (mirror of (1) with the
 *       reference's swapped constants)                             -> :229-269
 *   (4) neither: new entity, both sides from the base relations    -> :270-285 */
static int plan_join(predicate *pred, uint32_t *relations, DArray *entities, join_plan *plan)
{
    relation_column *second = (relation_column *)pred->second;
    join_side *L = &plan->lhs, *R = &plan->rhs;
    L->binding = pred->first.relation;
    L->rel = relations[L->binding];
    L->col = (uint32_t)pred->first.column;
    L->source = NULL;
    R->binding = second->relation;
    R->rel = relations[R->binding];
    R->col = (uint32_t)second->column;
    R->source = NULL;

    if (L->rel == R->rel && L->col == R->col) {
        plan->kind = DO_NOTHING;
        return 0;
    }

    DArray *current = DArray_count(entities) == 0 ? push_entity(entities) : *(DArray **)DArray_last(entities);
    if (current == NULL) return -1;

    const ssize_t li = relation_exists_current(current, L->rel, L->binding);
    const ssize_t ri = relation_exists_current(current, R->rel, R->binding);

    if (li != -1 && ri != -1) {
        L->source = (mid_result *)DArray_get(current, li);
        R->source = (mid_result *)DArray_get(current, ri);
        plan->kind = SCAN_JOIN;
    } else if (li != -1 || ri != -1) {
        /* `in` is the side found in the current entity, `out` the other one */
        const int lhs_in = li != -1;
        join_side *in = lhs_in ? L : R, *out = lhs_in ? R : L;
        in->source = (mid_result *)DArray_get(current, lhs_in ? li : ri);
        const int in_sorted = in->source->last_column_sorted == (int32_t)in->col;

        exists_info elsewhere = relation_exists(entities, out->rel, out->binding);
        if (elsewhere.index == -1) {
            /* other side straight from its base relation */
            if (in_sorted) {
                plan->kind = lhs_in ? JOIN_SORT_RHS : JOIN_SORT_LHS;
            } else {
                in->source->last_column_sorted = (int32_t)in->col;
                plan->kind = CLASSIC_JOIN;
            }
        } else {
            out->source = entry_at(entities, elsewhere);
            if (lhs_in) {
                const int out_sorted = out->source->last_column_sorted == (int32_t)out->col;
                plan->kind = (in_sorted && out_sorted) ? SCAN_JOIN
                             : in_sorted               ? JOIN_SORT_RHS
                             : out_sorted              ? JOIN_SORT_LHS
                                                       : CLASSIC_JOIN;
            } else {
                /* src/join.c:253-267: the rhs-sorted case answers JOIN_SORT_RHS and
                 * the third test looks at the *rhs* entry with the lhs column */
                const int out_sorted = out->source->last_column_sorted == (int32_t)out->col;
                const int in_has_lhs_col = in->source->last_column_sorted == (int32_t)L->col;
                plan->kind = (in_sorted && out_sorted) ? SCAN_JOIN
                             : in_sorted               ? JOIN_SORT_RHS
                             : in_has_lhs_col          ? JOIN_SORT_LHS
                                                       : CLASSIC_JOIN;
            }
        }
    } else {
        if (push_entity(entities) == NULL) return -1;
        plan->kind = (R->rel != L->rel || L->binding != R->binding) ? CLASSIC_JOIN : SCAN_JOIN;
    }
    return 0;
}

/* A base run that is sorted right after its build: built and sorted in one engine call, which can start the
 * sort from the column.  The reference to that entry is weak because the plain-C stand-in engine of the host
 * layer's CPU tests (tests/c/mock_engine.c) does not define it; libqce_b200 always does.  Without it the run is
 * built, then sorted -- which is what the entry returns. */
#pragma weak qce_build_sorted_tuples_base
static int build_sorted_base(uint32_t rel, uint32_t col, qce_tuples **out)
{
    if (qce_build_sorted_tuples_base) return qce_build_sorted_tuples_base(rel, col, out);
    if (qce_build_tuples_base(rel, col, out) != 0) return -1;
    if (qce_sort_tuples(*out) == 0) return 0;
    qce_tuples_free(*out);
    *out = NULL;
    return -1;
}

/* sorted: the side is sorted right after its build */
static int build_side(const join_side *s, int sorted, qce_tuples **out)
{
    if (s->source) {
        if (qce_build_tuples_rowids(s->rel, s->col, s->source->payloads, out) != 0) return -1;
        return sorted ? qce_sort_tuples(*out) : 0;
    }
    return sorted ? build_sorted_base(s->rel, s->col, out) : qce_build_tuples_base(s->rel, s->col, out);
}

static int require_sorted(const qce_tuples *t, const char *which)
{
    int sorted = 0;
    if (qce_tuples_is_sorted(t, &sorted) != 0) return -1;
    if (!sorted) {
        log_err("%s side of a JOIN_SORT merge is not in key order; the reference's result is "
                "order-dependent here (outside the parity-defined query class), query refused",
                which);
        return -1;
    }
    return 0;
}

/* Run the planned join on the device: res->results[] = aligned row-id columns. */
static int run_join(const join_plan *plan, join_result *res)
{
    qce_tuples *tl = NULL, *tr = NULL;
    int rc = -1;

    if (plan->kind == SCAN_JOIN) {
        const join_side *L = &plan->lhs, *R = &plan->rhs;
        if (L->source == NULL && R->source == NULL)
            rc = qce_scan_join_base(L->rel, L->col, R->rel, R->col, &res->results[0], &res->results[1]);
        else if (L->source != NULL && R->source != NULL)
            rc = qce_scan_join(L->rel, L->col, L->source->payloads, R->rel, R->col, R->source->payloads,
                               &res->results[0], &res->results[1]);
        if (rc != 0) log_err("scan join failed: %s", qce_last_error());
        return rc;
    }

    const int sort_lhs = plan->kind == CLASSIC_JOIN || plan->kind == JOIN_SORT_LHS;
    const int sort_rhs = plan->kind == CLASSIC_JOIN || plan->kind == JOIN_SORT_RHS;
    check(build_side(&plan->lhs, sort_lhs, &tl) == 0 && build_side(&plan->rhs, sort_rhs, &tr) == 0,
          "Couldn't allocate relations: %s", qce_last_error());
    /* with an empty side the pointer walk of src/join.c:342 never starts: the
     * result is empty whatever the order of the other side */
    const int trivially_empty = qce_tuples_count(tl) == 0 || qce_tuples_count(tr) == 0;
    int outer_in_order = 1;
    if (!sort_lhs && !trivially_empty) {
        /* JOIN_SORT_RHS trusts the lhs to be in key order.  When it is not (the
         * asymmetric tests of src/join.c:253-267), the reference's walk is still a
         * function of the data -- qce_merge_join_walk computes it. */
        check(qce_tuples_is_sorted(tl, &outer_in_order) == 0, "%s", qce_last_error());
    }
    if (!sort_rhs && !trivially_empty) {
        check(require_sorted(tr, "right") == 0, "Join failed!");
    }
    if (outer_in_order) {
        check(qce_merge_join(tl, tr, &res->results[0], &res->results[1], NULL, NULL) == 0, "merge join failed: %s",
              qce_last_error());
    } else {
        check(qce_merge_join_walk(tl, tr, &res->results[0], &res->results[1]) == 0, "merge join failed: %s",
              qce_last_error());
    }
    rc = 0;

error:
    qce_tuples_free(tl);
    qce_tuples_free(tr);
    return rc;
}

/* The distinct (rowid_lhs,rowid_rhs) pairs are only ever consumed by a
 * bystander re-join, so they are computed the first time one is needed. */
static int need_distinct(join_result *res)
{
    if (res->non_duplicates[0] != NULL) return 0;
    if (qce_distinct_pairs(res->results[0], res->results[1], &res->non_duplicates[0], &res->non_duplicates[1]) != 0) {
        log_err("distinct pairs failed: %s", qce_last_error());
        return -1;
    }
    return 0;
}

/* fix_all_mid_results, src/join.c:486-505: every other column of the entity
 * (test is on the relation id, :495) is re-joined against the distinct pairs'
 * `side`, then the joined binding's entry is replaced. */
static int replace_and_rejoin(join_result *res, DArray *entities, exists_info where, const join_plan *plan,
                              mid_result fresh, int side)
{
    DArray *entity = *(DArray **)DArray_get(entities, where.mid_result);
    mid_result *joined = (mid_result *)DArray_get(entity, where.index);

    for (size_t i = 0; i < DArray_count(entity); i++) {
        mid_result *bystander = (mid_result *)DArray_get(entity, i);
        if (bystander->relation == plan->lhs.rel || bystander->relation == plan->rhs.rel) continue;
        if (qce_join_elide_active() && entity_rejoined(entity)) {
            /* a faithful replay on top of an elided one would pair columns the reference has in another order */
            qce_join_elide_raise();
            return -1;
        }
        mark_rejoined(entity);
        if (need_distinct(res) != 0) return -1;
        struct qce_rowids *rejoined = NULL;
        if (qce_rejoin(res->non_duplicates[side], joined->payloads, bystander->payloads, &rejoined) != 0) {
            log_err("bystander re-join failed: %s", qce_last_error());
            return -1;
        }
        qce_rowids_free(bystander->payloads);
        bystander->payloads = rejoined;
    }
    qce_rowids_free(joined->payloads);
    *joined = fresh;
    return 0;
}

static void fatal_inconsistent(void)
{
    log_err("Something went really wrong");
    qce_fatal(); /* src/join.c:563,601,610,620: exit(EXIT_FAILURE), after the earlier queries' stdout */
}

/* update_mid_results, src/join.c:507-628. */
static int install_results(join_result *res, DArray *entities, const join_plan *plan)
{
    mid_result fresh[2];
    const join_side *sides[2] = {&plan->lhs, &plan->rhs};
    for (int s = 0; s < 2; s++) {
        fresh[s].relation = sides[s]->rel;
        fresh[s].predicate_id = sides[s]->binding;
        fresh[s].last_column_sorted = (int32_t)sides[s]->col;
        fresh[s].payloads = res->results[s];
    }

    if (plan->kind == SCAN_JOIN) {
        /* only the row-id columns are swapped in; bystanders and the sorted
         * column marker stay as they were (:607-627) */
        mid_result *touched[2] = {NULL, NULL};
        for (int s = 0; s < 2; s++) {
            exists_info where = relation_exists(entities, sides[s]->rel, sides[s]->binding);
            if (where.index == -1) fatal_inconsistent();
            mid_result *entry = entry_at(entities, where);
            if (entry->payloads != res->results[0] && entry->payloads != res->results[1])
                qce_rowids_free(entry->payloads); /* the reference leaks the old array */
            entry->payloads = res->results[s];
            touched[s] = entry;
        }
        /* both sides on one binding (a predicate like 0.1=0.2): the entry now holds results[1] and results[0],
         * the same row ids, belongs to nobody -- 4 bytes per surviving row were lost per query */
        if (touched[0] == touched[1] && res->results[0] != res->results[1]) {
            qce_rowids_free(res->results[0]);
            res->results[0] = res->results[1];
        }
        return 0;
    }

    /* order and strictness per kind:
     *   CLASSIC        lhs then rhs, each pushed if new else re-joined
     *   JOIN_SORT_LHS  lhs pushed or plainly replaced, then rhs must exist and is re-joined
     *   JOIN_SORT_RHS  rhs pushed or plainly replaced, then lhs must exist and is re-joined */
    const int first = plan->kind == JOIN_SORT_RHS ? 1 : 0;
    for (int step = 0; step < 2; step++) {
        const int s = step == 0 ? first : 1 - first;
        const int plain_replace = plan->kind != CLASSIC_JOIN && step == 0;
        const int must_exist = plan->kind != CLASSIC_JOIN && step == 1;
        exists_info where = relation_exists(entities, sides[s]->rel, sides[s]->binding);
        if (where.index == -1) {
            if (must_exist) fatal_inconsistent();
            DArray *last = *(DArray **)DArray_last(entities);
            DArray_push(last, &fresh[s]);
        } else if (plain_replace) {
            mid_result *entry = entry_at(entities, where);
            qce_rowids_free(entry->payloads);
            *entry = fresh[s];
        } else if (replace_and_rejoin(res, entities, where, plan, fresh[s], s) != 0) {
            return -1;
        }
    }
    return 0;
}

/* ---- the elided join (see the top of this file) ----------------------------------------------- */
static DArray *entity_of(DArray *entities, const mid_result *m)
{
    for (size_t e = 0; e < DArray_count(entities); e++) {
        DArray *entity = *(DArray **)DArray_get(entities, e);
        for (size_t j = 0; j < DArray_count(entity); j++)
            if ((const mid_result *)DArray_get(entity, j) == m) return entity;
    }
    return NULL;
}
static int has_bystanders(DArray *entity, const join_plan *plan)
{
    for (size_t i = 0; i < DArray_count(entity); i++) {
        const mid_result *m = (const mid_result *)DArray_get(entity, i);
        if (m->relation != plan->lhs.rel && m->relation != plan->rhs.rel) return 1;
    }
    return 0;
}

/* 1: the join ran in elided mode and its results are installed; 0: not applicable, take the
 * faithful path; QCE_JOIN_UNSAFE: elided mode can no longer vouch for the reference's result. */
static int elided_join(const join_plan *plan, DArray *entities)
{
    const join_side *sides[2] = {&plan->lhs, &plan->rhs};
    DArray *ent[2] = {NULL, NULL};
    int bys[2] = {0, 0};
    for (int s = 0; s < 2; s++)
        if (sides[s]->source) {
            ent[s] = entity_of(entities, sides[s]->source);
            bys[s] = ent[s] ? has_bystanders(ent[s], plan) : 0;
        }
    const int rej0 = ent[0] && entity_rejoined(ent[0]), rej1 = ent[1] && entity_rejoined(ent[1]);

    if (plan->kind == SCAN_JOIN) /* positional: the order inside a re-joined entity differs from the reference's */
        return (rej0 || rej1) ? QCE_JOIN_UNSAFE : 0;
    if (!bys[0] && !bys[1]) {
        /* no column is re-joined; but a JOIN_SORT_* trusts the order of a column the reference has re-ordered */
        if (plan->kind == JOIN_SORT_RHS && rej0) return QCE_JOIN_UNSAFE;
        if (plan->kind == JOIN_SORT_LHS && rej1) return QCE_JOIN_UNSAFE;
        return 0;
    }
    /* exactly one side comes from an entity with bystanders; the other one is a base relation */
    const int s = bys[0] ? 0 : 1, o = 1 - s;
    if (bys[o] || sides[o]->source != NULL) return QCE_JOIN_UNSAFE;
    const int rejoined = s == 0 ? rej0 : rej1;
    if (rejoined && (s != 0 || plan->kind != CLASSIC_JOIN)) return QCE_JOIN_UNSAFE; /* the match counts are per outer tuple */
    if (plan->kind == JOIN_SORT_RHS && s != 0) return QCE_JOIN_UNSAFE;
    if (plan->kind == JOIN_SORT_LHS && s != 1) return QCE_JOIN_UNSAFE;

    qce_tuples *t[2] = {NULL, NULL};
    struct qce_rowids *out[2] = {NULL, NULL}, *fresh_ids = NULL;
    int rc = -1;
    if (qce_build_tuples_positions(sides[s]->rel, sides[s]->col, sides[s]->source->payloads, &t[s]) != 0)
        return 0; /* keys >= 2^32: the faithful path handles them */
    {
        /* every column that will follow the positions (the joined one and the bystanders, by the
         * relation-id test of src/join.c:495); with several ranks they travel with the tuples */
        const struct qce_rowids *cols[8];
        uint32_t nc = 0;
        for (size_t i = 0; i < DArray_count(ent[s]); i++) {
            const mid_result *m = (const mid_result *)DArray_get(ent[s], i);
            const int joined = m == sides[s]->source;
            if (!joined && (m->relation == plan->lhs.rel || m->relation == plan->rhs.rel)) continue;
            if (nc == 6 || qce_rowids_count(m->payloads) < qce_rowids_count(sides[s]->source->payloads)) { rc = QCE_JOIN_UNSAFE; goto done; }
            cols[nc++] = m->payloads;
        }
        if (qce_tuples_attach(t[s], nc, cols) != 0) { rc = QCE_JOIN_UNSAFE; goto done; }
    }
    /* the base side is always sorted */
    if (build_sorted_base(sides[o]->rel, sides[o]->col, &t[o]) != 0) {
        log_err("Couldn't build and sort a relation: %s", qce_last_error());
        goto done;
    }
    if (plan->kind == CLASSIC_JOIN) {
        if (qce_sort_tuples(t[s]) != 0) { log_err("sort failed: %s", qce_last_error()); goto done; }
    } else {
        /* the entity side is trusted to be in key order (src/join.c:197-204): only vouched for when it is */
        int sorted = 0;
        if (qce_tuples_count(t[s]) && qce_tuples_count(t[o])) {
            if (qce_tuples_is_sorted(t[s], &sorted) != 0) { log_err("%s", qce_last_error()); goto done; }
            if (!sorted) { rc = QCE_JOIN_UNSAFE; goto done; }
        }
    }
    uint32_t lo = 0, hi = 0;
    if (qce_merge_join_stats(t[0], t[1], &out[0], &out[1], &lo, &hi) != 0) { log_err("merge join failed: %s", qce_last_error()); goto done; }
    if (rejoined && lo != hi && qce_tuples_count(t[0]) && qce_tuples_count(t[1])) { rc = QCE_JOIN_UNSAFE; goto done; }

    /* out[s] holds POSITIONS in the entity: every column of the entity follows them */
    for (size_t i = 0; i < DArray_count(ent[s]); i++) {
        mid_result *m = (mid_result *)DArray_get(ent[s], i);
        const int joined = m == sides[s]->source;
        if (!joined && (m->relation == plan->lhs.rel || m->relation == plan->rhs.rel)) continue; /* src/join.c:495: by relation id */
        if (qce_rowids_count(m->payloads) < qce_rowids_count(sides[s]->source->payloads)) { rc = QCE_JOIN_UNSAFE; goto done; }
    }
    for (size_t i = 0; i < DArray_count(ent[s]); i++) {
        mid_result *m = (mid_result *)DArray_get(ent[s], i);
        const int joined = m == sides[s]->source;
        if (!joined && (m->relation == plan->lhs.rel || m->relation == plan->rhs.rel)) continue;
        struct qce_rowids *g = NULL;
        if (qce_rowids_gather(m->payloads, out[s], &g) != 0) { log_err("gather failed: %s", qce_last_error()); goto done; }
        if (joined) { fresh_ids = g; continue; } /* installed last: it still indexes nothing else */
        qce_rowids_free(m->payloads);
        m->payloads = g;
    }
    {
        mid_result *joined = sides[s]->source;
        qce_rowids_free(joined->payloads);
        joined->payloads = fresh_ids;
        joined->last_column_sorted = (int32_t)sides[s]->col;
        fresh_ids = NULL;
        mid_result other;
        other.relation = sides[o]->rel;
        other.predicate_id = sides[o]->binding;
        other.last_column_sorted = (int32_t)sides[o]->col;
        other.payloads = out[o];
        out[o] = NULL;
        DArray *last = *(DArray **)DArray_last(entities);
        DArray_push(last, &other);
    }
    mark_rejoined(ent[s]);
    rc = 1;

done:
    qce_tuples_free(t[0]);
    qce_tuples_free(t[1]);
    qce_rowids_free(out[0]);
    qce_rowids_free(out[1]);
    qce_rowids_free(fresh_ids);
    return rc;
}

int execute_join(predicate *pred, uint32_t *relations, DArray *metadata_arr, DArray *mid_results_array)
{
    (void)metadata_arr;
    join_plan plan;
    join_result res = {{NULL, NULL}, {NULL, NULL}};

    if (plan_join(pred, relations, mid_results_array, &plan) != 0) return -1;
    if (plan.kind == DO_NOTHING) return 0;
    debug("join kind %d", plan.kind);
    if (qce_join_elide_active()) {
        const int r = elided_join(&plan, mid_results_array);
        if (r == QCE_JOIN_UNSAFE) { qce_join_elide_raise(); return QCE_JOIN_UNSAFE; }
        if (r != 0) return r == 1 ? 0 : -1;
    }

    if (run_join(&plan, &res) != 0) goto error;
    if (install_results(&res, mid_results_array, &plan) != 0) goto error_installed;

    qce_rowids_free(res.non_duplicates[0]);
    qce_rowids_free(res.non_duplicates[1]);
    return 0;

error:
    qce_rowids_free(res.results[0]);
    qce_rowids_free(res.results[1]);
error_installed:
    qce_rowids_free(res.non_duplicates[0]);
    qce_rowids_free(res.non_duplicates[1]);
    return -1;
}
