/*
 * TEST INFRASTRUCTURE — risk6_vector.c: the six-player search with a six-seat value vector (SIXPLAYER.md §2, "value vector"), the
 * checker of az_mcts6_* over a network with six value outputs or with AZ_EVAL_PSEUDO6.  An evaluator returns value[6] relative to the
 * leaf's seat to move L: value[k] belongs to seat (L + k) % 6.  A path node whose mover is s receives value[(s - L + 6) % 6] in
 * Q = (N * Q + val) / (N + 1); a finished game backs up with the scalar rule (1 for the winner's nodes, -1/5 for the others, 0 after
 * a draw); the node's stored value is component 0.  Everything else is r6l_search: K descents per round in the lockstep schedule with
 * the active_N rule, completion in descent order, a duplicate leaf not inserted again but its own vector backed up.
 *
 * It builds on risk6_lockstep.c and risk6_oracle.c unchanged (included here, so the rules, the table, the selection and the scalar
 * backup are those files' own code).  The vector evaluator is reached through the table's scalar evaluator slot: a trampoline keeps
 * the last vector beside the table and hands component 0 to expand6.  Built as its own library by oracle/vector6.py; never linked
 * into the product.
 */
#include "risk6_lockstep.c"

typedef void (*r6v_eval_fn)(const r6_state* s, float policy[RO_MOVES], float value[R6_PLAYERS], void* user);

typedef struct r6v_mcts {
    r6l_mcts* l;
    r6v_eval_fn eval;
    void* user;
    float last[R6_PLAYERS];              /* the vector of the last evaluation */
} r6v_mcts;

/* the pseudo evaluator with az_pn_value6 (AZ_EVAL_PSEUDO6): r6_eval_pseudo's policy, value[k] = az_pn_value6(key, k) */
void r6v_eval_pseudo6(const r6_state* s, float policy[RO_MOVES], float value[R6_PLAYERS], void* user)
{
    (void)user;
    const uint64_t key = pn_key6(s);
    for (int i = 0; i < RO_MOVES; ++i) policy[i] = az_pn_policy(key, i);
    for (int k = 0; k < R6_PLAYERS; ++k) value[k] = az_pn_value6(key, k);
}

static void trampoline(const r6_state* s, float policy[RO_MOVES], float* value, void* user)
{
    r6v_mcts* v = (r6v_mcts*)user;
    v->eval(s, policy, v->last, v->user);
    *value = v->last[0];
}

r6v_mcts* r6v_new(r6v_eval_fn eval, void* user)
{
    r6v_mcts* v = (r6v_mcts*)calloc(1, sizeof *v);
    v->eval = eval ? eval : r6v_eval_pseudo6;
    v->user = user;
    v->l = r6l_new(trampoline, v);
    return v;
}
void r6v_free(r6v_mcts* v) { if (v) { r6l_free(v->l); free(v); } }
int r6v_table_size(const r6v_mcts* v) { return v->l->m->n_nodes; }
uint64_t r6v_vl_skips(const r6v_mcts* v) { return v->l->vl_skips; }
uint64_t r6v_active_total(const r6v_mcts* v) { return r6l_active_total(v->l); }

/* backup_l with the per-seat rule: the node of mover s receives vec[(s - seat + 6) % 6], seat = the leaf's seat to move */
static void backup_v(r6l_mcts* l, const r6l_descent* d, const float vec[R6_PLAYERS], int seat)
{
    for (int k = d->len - 1; k >= 0; --k) {
        r6_node* n = &l->m->nodes[d->node[k]];
        const int mv = d->mv[k];
        float val = vec[(d->mover[k] - seat + R6_PLAYERS) % R6_PLAYERS];
        if (n->N[mv] == 0) n->Q[mv] = val; else n->Q[mv] = ((float)n->N[mv] * n->Q[mv] + val) / (float)(n->N[mv] + 1);
        n->N[mv]++; n->sumN++;
        l->active[d->node[k]][mv]--;
    }
}

/* r6l_search with the per-seat backup; RO_ERR_ILLEGAL_ACTION when K < 1 or K does not divide the simulation count */
int r6v_search(r6v_mcts* v, const r6_state* root, const ro_rules* r, uint64_t seed, uint32_t game, uint32_t ply, int K,
               uint32_t N[RO_MOVES], float Q[RO_MOVES], float P[RO_MOVES], float pi[RO_MOVES], uint32_t* sumN, float* root_value)
{
    r6l_mcts* l = v->l;
    const int count = r->mcts_simulations - (r->mcts_simulations % r->threads_per_mcts);
    if (K < 1 || count % K != 0) return RO_ERR_ILLEGAL_ACTION;
    r6_mcts* m = l->m;
    m->n_nodes = 0;
    float v0; expand_l(l, root, r6_valid_moves(root, r), &v0);
    r6l_descent* ds = (r6l_descent*)malloc(sizeof(r6l_descent) * (size_t)K);
    int rc = RO_OK;
    for (int round = 0; round < count / K && rc == RO_OK; ++round) {
        for (int j = 0; j < K && rc == RO_OK; ++j) {                  /* selection, in descent order (r6l_search) */
            r6l_descent* d = &ds[j];
            d->len = 0; d->pending = 0;
            r6_state s = *root; uint32_t die = 0;
            const uint32_t sim = (uint32_t)(round * K + j);
            for (;;) {
                int gs = r6_game_status(&s, r);
                if (gs != R6_NOT_ENDED) { backup_l(l, d, gs == R6_DRAW ? 0.0f : 1.0f, gs == R6_DRAW ? s.cur : gs); break; }
                uint64_t valid = r6_valid_moves(&s, r);
                int idx = find6(m, &s);
                if (idx < 0) { d->leaf = s; d->valid = valid; d->pending = 1; break; }
                if (d->len == R6L_PATH_MAX) { rc = RO_ERR_ILLEGAL_ACTION; break; }
                int mv = select_l(l, idx, r);
                int cur = s.cur;
                if (make_move_stream(&s, mv, r, seed, game, ply, sim, &die) != RO_OK) { rc = RO_ERR_ILLEGAL_ACTION; break; }
                d->node[d->len] = idx; d->mv[d->len] = (uint8_t)mv; d->mover[d->len] = (uint8_t)cur; d->len++;
            }
        }
        for (int j = 0; j < K && rc == RO_OK; ++j) {                  /* completion, in descent order: each leaf's own vector */
            r6l_descent* d = &ds[j];
            if (!d->pending) continue;
            float val;
            if (find6(m, &d->leaf) < 0) expand_l(l, &d->leaf, d->valid, &val);
            else { float policy[RO_MOVES]; m->eval(&d->leaf, policy, &val, m->user); m->evals++; }
            backup_v(l, d, v->last, d->leaf.cur);
        }
    }
    free(ds);
    if (rc != RO_OK) return rc;
    const r6_node* n = &m->nodes[find6(m, root)];                      /* root statistics exactly as r6_mcts_search */
    float sum = 0.0f;
    for (int i = 0; i < RO_MOVES; ++i) {
        int ok = (int)((n->valid >> i) & 1);
        N[i] = ok ? n->N[i] : 0; Q[i] = ok ? n->Q[i] : 0.0f; P[i] = ok ? n->P[i] : 0.0f;
        pi[i] = ok ? (float)n->N[i] : 0.0f;
        if (ok) sum += pi[i];
    }
    for (int i = 0; i < RO_MOVES; ++i) pi[i] /= sum;
    *sumN = n->sumN; *root_value = n->value;
    return RO_OK;
}
