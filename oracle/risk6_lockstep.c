/*
 * TEST INFRASTRUCTURE — risk6_lockstep.c: the six-player search with K descents per round (SIXPLAYER.md §2, "descents per tree"),
 * the checker of az_mcts6_* with az_rules.concurrent_descents = K.  The six-player counterpart of ro_mcts_search_lockstep
 * (risk_oracle.c): descent j of round r uses the dice stream sim = r * K + j and selects after descents 0..j-1 with
 * getNextBestMoveAndSetVisited's active_N rule (alphazero_mcts.cpp:91-111); the pending leaves are expanded and backed up in descent
 * order, a duplicate is not inserted again but its value is backed up (StateSimulationsStorage::add :203-215).
 *
 * It builds on risk6_oracle.c unchanged (included here, so the rules, the table and the evaluator are that file's own code) and keeps
 * the active_N marks in an array beside the table.  Built as its own library by oracle/lockstep6.py; never linked into the product.
 */
#include "risk6_oracle.c"

typedef struct r6l_mcts {
    r6_mcts* m;
    uint32_t (*active)[RO_MOVES];        /* active_N per node of m's table and move */
    int active_cap;
    uint64_t vl_skips, vl_duplicates;
} r6l_mcts;

r6l_mcts* r6l_new(r6_eval_fn eval, void* user)
{
    r6l_mcts* l = (r6l_mcts*)calloc(1, sizeof *l);
    l->m = r6_mcts_new(eval, user);
    return l;
}
void r6l_free(r6l_mcts* l) { if (l) { r6_mcts_free(l->m); free(l->active); free(l); } }
int r6l_table_size(const r6l_mcts* l) { return l->m->n_nodes; }
uint64_t r6l_vl_skips(const r6l_mcts* l) { return l->vl_skips; }
uint64_t r6l_vl_duplicates(const r6l_mcts* l) { return l->vl_duplicates; }
uint64_t r6l_active_total(const r6l_mcts* l)
{
    uint64_t t = 0;
    for (int i = 0; i < l->m->n_nodes; ++i) for (int k = 0; k < RO_MOVES; ++k) t += l->active[i][k];
    return t;
}

/* expand6 plus a cleared active_N row for the new node */
static void expand_l(r6l_mcts* l, const r6_state* s, uint64_t valid, float* value_out)
{
    expand6(l->m, s, valid, value_out);
    if (l->m->n_nodes > l->active_cap) {
        l->active_cap = l->m->cap;
        l->active = (uint32_t(*)[RO_MOVES])realloc(l->active, sizeof *l->active * (size_t)l->active_cap);
    }
    memset(l->active[l->m->n_nodes - 1], 0, sizeof *l->active);
}

/* getNextBestMoveAndSetVisited with the active_N rule, as select_move in risk_oracle.c */
static int select_l(r6l_mcts* l, int idx, const ro_rules* r)
{
    const r6_node* n = &l->m->nodes[idx];
    uint32_t* act = l->active[idx];
    int best = -1, dup = -1; float best_u = -INFINITY, dup_u = -INFINITY;
    for (int i = 0; i < RO_MOVES; ++i) {
        if (!((n->valid >> i) & 1)) continue;
        float noiseP = (1 - r->dir_noise_epsi) * n->P[i] + r->dir_noise_epsi * r->dir_noise_value;
        float v = noiseP * r->cpuct * sqrtf(1.0f + (float)n->sumN);
        float u = n->Q[i] + (v / (1.0f + (float)n->N[i]));
        if (u > best_u) {
            if (n->N[i] == 0 && act[i] == 1) { l->vl_skips++; if (u > dup_u) { dup_u = u; dup = i; } }
            else { best_u = u; best = i; }
        }
    }
    if (best < 0) { best = dup; l->vl_duplicates++; }
    act[best]++;
    return best;
}

#define R6L_PATH_MAX 1024
typedef struct r6l_descent {
    int node[R6L_PATH_MAX]; uint8_t mv[R6L_PATH_MAX], mover[R6L_PATH_MAX];
    int len, pending;
    r6_state leaf; uint64_t valid;
} r6l_descent;

/* addValue up the path with the six-seat rule (search6's arithmetic); every step takes the descent's active_N mark off its move */
static void backup_l(r6l_mcts* l, const r6l_descent* d, float v, int seat)
{
    for (int k = d->len - 1; k >= 0; --k) {
        r6_node* n = &l->m->nodes[d->node[k]];
        const int mv = d->mv[k];
        float val = d->mover[k] == seat ? v : -v / 5.0f;
        if (n->N[mv] == 0) n->Q[mv] = val; else n->Q[mv] = ((float)n->N[mv] * n->Q[mv] + val) / (float)(n->N[mv] + 1);
        n->N[mv]++; n->sumN++;
        l->active[d->node[k]][mv]--;
    }
}

/* K descents per round; K = 1 is r6_mcts_search.  RO_ERR_ILLEGAL_ACTION when K < 1 or K does not divide the simulation count. */
int r6l_search(r6l_mcts* l, const r6_state* root, const ro_rules* r, uint64_t seed, uint32_t game, uint32_t ply, int K,
               uint32_t N[RO_MOVES], float Q[RO_MOVES], float P[RO_MOVES], float pi[RO_MOVES], uint32_t* sumN, float* root_value)
{
    const int count = r->mcts_simulations - (r->mcts_simulations % r->threads_per_mcts);
    if (K < 1 || count % K != 0) return RO_ERR_ILLEGAL_ACTION;
    r6_mcts* m = l->m;
    m->n_nodes = 0;
    float v0; expand_l(l, root, r6_valid_moves(root, r), &v0);
    r6l_descent* ds = (r6l_descent*)malloc(sizeof(r6l_descent) * (size_t)K);
    int rc = RO_OK;
    for (int round = 0; round < count / K && rc == RO_OK; ++round) {
        for (int j = 0; j < K && rc == RO_OK; ++j) {                  /* selection, in descent order */
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
        for (int j = 0; j < K && rc == RO_OK; ++j) {                  /* completion, in descent order */
            r6l_descent* d = &ds[j];
            if (!d->pending) continue;
            float v;
            if (find6(m, &d->leaf) < 0) expand_l(l, &d->leaf, d->valid, &v);
            else { float policy[RO_MOVES]; m->eval(&d->leaf, policy, &v, m->user); m->evals++; }
            backup_l(l, d, v, d->leaf.cur);
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
