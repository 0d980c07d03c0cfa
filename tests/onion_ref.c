/* onion_ref.c -- TEST INFRASTRUCTURE: a serial restatement of the onion decomposition (networkx.onion_layers) in
 * O(n + m + max degree), so that graphs far too large for networkx (which sorts every remaining vertex once per
 * layer) can be checked.  tests/onion_ref.py compiles and wraps it; tests/test_onion_cpu.py pins it to networkx.
 *
 * Input: n vertices and E simple undirected edges (u, v), no loops, no duplicates.
 * Output: layer[v] (1-based) and core[v] (the level k the vertex is removed at).  Returns the number of layers, or -1
 * when memory runs out.
 *
 * Degree-0 vertices form layer 1 when there are any.  Then k starts at 1; each level sets k to max(k, smallest
 * remaining degree); its first layer is every remaining vertex of degree k, and each further layer is every vertex
 * whose degree fell from above k to at most k while the previous layer was removed.  The smallest remaining degree
 * is found with lazy buckets: a vertex is pushed into bucket d whenever its degree becomes d > k, and stale entries
 * (removed, or degree changed since) are skipped. */
#include <stdint.h>
#include <stdlib.h>

long long onion_ref(uint32_t n, const uint32_t *eu, const uint32_t *ev, uint64_t E, uint32_t *layer, int32_t *core) {
    long long rc = -1;
    uint64_t *ptr = calloc((size_t)n + 1, sizeof(uint64_t));
    uint32_t *adj = malloc((2 * E + 1) * sizeof(uint32_t));
    int64_t *deg = malloc(((size_t)n + 1) * sizeof(int64_t));
    uint8_t *gone = calloc((size_t)n + 1, 1);
    uint32_t *cur = malloc(((size_t)n + 1) * sizeof(uint32_t)), *nxt = malloc(((size_t)n + 1) * sizeof(uint32_t));
    /* lazy buckets: at most n initial entries + one per decrement */
    const uint64_t cap = (uint64_t)n + 2 * E + 1;
    uint32_t *b_v = malloc(cap * sizeof(uint32_t));
    uint64_t *b_next = malloc(cap * sizeof(uint64_t));
    uint64_t *head = NULL;
    uint64_t b_used = 0, maxdeg = 0;
    if (!ptr || !adj || !deg || !gone || !cur || !nxt || !b_v || !b_next) goto out;
    for (uint64_t e = 0; e < E; ++e) { ptr[eu[e] + 1]++; ptr[ev[e] + 1]++; }
    for (uint32_t v = 0; v < n; ++v) ptr[v + 1] += ptr[v];
    {
        uint64_t *fill = malloc(((size_t)n + 1) * sizeof(uint64_t));
        if (!fill) goto out;
        for (uint32_t v = 0; v <= n; ++v) fill[v] = ptr[v];
        for (uint64_t e = 0; e < E; ++e) { adj[fill[eu[e]]++] = ev[e]; adj[fill[ev[e]]++] = eu[e]; }
        free(fill);
    }
    for (uint32_t v = 0; v < n; ++v) {
        deg[v] = (int64_t)(ptr[v + 1] - ptr[v]);
        if ((uint64_t)deg[v] > maxdeg) maxdeg = (uint64_t)deg[v];
    }
    head = malloc((maxdeg + 2) * sizeof(uint64_t));
    if (!head) goto out;
    for (uint64_t d = 0; d <= maxdeg + 1; ++d) head[d] = UINT64_MAX;
#define PUSH(v, d) do { b_v[b_used] = (v); b_next[b_used] = head[d]; head[d] = b_used++; } while (0)

    uint32_t L = 0, left = n;
    {   /* layer 1: the isolated vertices */
        uint32_t iso = 0;
        for (uint32_t v = 0; v < n; ++v)
            if (deg[v] == 0) { layer[v] = 1; core[v] = 0; gone[v] = 1; ++iso; }
        if (iso) { L = 1; left -= iso; }
    }
    for (uint32_t v = n; v-- > 0;)
        if (!gone[v]) PUSH(v, (uint64_t)deg[v]);
    int64_t k = 1;
    uint64_t d = 1;
    while (left) {
        /* the smallest remaining degree: the first bucket >= k with a live entry */
        uint32_t nc = 0;
        for (; d <= maxdeg && nc == 0; ++d) {
            if ((int64_t)d < k) continue;
            for (uint64_t i = head[d]; i != UINT64_MAX; i = b_next[i]) {
                const uint32_t v = b_v[i];
                if (!gone[v] && deg[v] == (int64_t)d) { cur[nc++] = v; gone[v] = 1; }
            }
            head[d] = UINT64_MAX;
            if (nc) k = (int64_t)d;
        }
        if (nc == 0) goto out;   /* unreachable for a consistent graph */
        while (nc) {
            ++L;
            for (uint32_t i = 0; i < nc; ++i) { layer[cur[i]] = L; core[cur[i]] = (int32_t)k; }
            left -= nc;
            uint32_t nn = 0;
            for (uint32_t i = 0; i < nc; ++i) {
                const uint32_t v = cur[i];
                for (uint64_t e = ptr[v]; e < ptr[v + 1]; ++e) {
                    const uint32_t u = adj[e];
                    if (gone[u]) continue;
                    const int64_t old = deg[u]--;
                    if (old == k + 1) nxt[nn++] = u;
                    else if (old > k + 1) PUSH(u, (uint64_t)(old - 1));
                }
            }
            for (uint32_t i = 0; i < nn; ++i) gone[nxt[i]] = 1;   /* the next layer is removed at once */
            uint32_t *t = cur; cur = nxt; nxt = t;
            nc = nn;
        }
        d = (uint64_t)k + 1;
    }
    rc = L;
out:
    free(ptr); free(adj); free(deg); free(gone); free(cur); free(nxt); free(b_v); free(b_next); free(head);
    return rc;
}
