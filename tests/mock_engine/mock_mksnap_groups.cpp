// mock_mksnap_groups.cpp -- TEST INFRASTRUCTURE ONLY: the CPU mock of libmksnap (mock_mksnap.cpp, included unchanged)
// plus the grouped-session calls libmkhost makes for a batch commit with per-layer tables (MKHOST_LAYER_TABLES):
// mksnap_begin_groups / mksnap_arena_submit_groups / mksnap_get_group_results (DESIGN.md section 3c).  The plain
// begin / submit / finish / destroy of the included mock are wrapped: the wrappers keep, per handle, the group of every
// chunk and build each group's table and root at finish with the oracle (oracle/mkoracle.c), exactly as an ungrouped
// session of that group's files would.  Like the mock it extends, it is never loaded by the product.
#define mksnap_begin mock_plain_begin
#define mksnap_arena_submit mock_plain_arena_submit
#define mksnap_finish mock_plain_finish
#define mksnap_destroy mock_plain_destroy
#include "mock_mksnap.cpp"
#undef mksnap_begin
#undef mksnap_arena_submit
#undef mksnap_finish
#undef mksnap_destroy

namespace {

struct GroupState {
    uint32_t n_groups = 0, open_group = 0;
    std::vector<uint32_t> chunk_group;        // per chunk digest of the session
    std::vector<uint8_t> open_bytes;          // pieces of a file that spans submits (to count its chunks)
    std::vector<mksnap_group_result> res;
};

std::map<const mksnap *, GroupState> g_groups; // handles in a grouped session

size_t count_cuts(const mksnap *h, const uint8_t *p, uint64_t n)
{
    mko_cdc_params prm;
    mko_cdc_default_params(&prm);
    if (h->cfg.cdc.min_size)
        memcpy(&prm, &h->cfg.cdc, sizeof prm);
    std::vector<uint64_t> ends((size_t)(n / prm.min_size) + 2);
    return mko_cdc_cuts(p, n, &prm, ends.data(), ends.size());
}

} // namespace

extern "C" {

int mksnap_begin(mksnap_t *h)
{
    g_groups.erase(h);
    return mock_plain_begin(h);
}

void mksnap_destroy(mksnap_t *h)
{
    g_groups.erase(h);
    mock_plain_destroy(h);
}

int mksnap_begin_groups(mksnap_t *h, uint32_t n_groups)
{
    if (!h)
        return MKSNAP_E_INVAL;
    if (n_groups == 0 || n_groups > 65536)
        return fail(h, MKSNAP_E_INVAL, "n_groups must be in [1, 65536]");
    const int rc = mksnap_begin(h);
    if (rc)
        return rc;
    GroupState &st = g_groups[h];
    st.n_groups = n_groups;
    st.res.assign(n_groups, mksnap_group_result{});
    return 0;
}

int mksnap_arena_submit(mksnap_t *h, int32_t arena_id, uint64_t used, const mksnap_extent *ext, uint64_t n_ext,
                        const mksnap_range *rng, uint64_t n_rng)
{
    if (h && g_groups.count(h))
        return fail(h, MKSNAP_E_STATE, "a grouped session takes mksnap_arena_submit_groups");
    return mock_plain_arena_submit(h, arena_id, used, ext, n_ext, rng, n_rng);
}

int mksnap_arena_submit_groups(mksnap_t *h, int32_t arena_id, uint64_t used, const mksnap_extent *ext, uint64_t n_ext,
                               const uint32_t *groups, const mksnap_range *rng, uint64_t n_rng)
{
    if (!h)
        return MKSNAP_E_INVAL;
    auto it = g_groups.find(h);
    if (it == g_groups.end())
        return fail(h, MKSNAP_E_STATE, "grouped submit in a session that mksnap_begin started");
    GroupState &st = it->second;
    if (n_ext && !groups)
        return fail(h, MKSNAP_E_INVAL, "null group table");
    if (arena_id < 0 || (size_t)arena_id >= h->arenas.size() || !h->acquired[arena_id] || used > h->arenas[arena_id].size())
        return mock_plain_arena_submit(h, arena_id, used, ext, n_ext, rng, n_rng); // its own error
    for (uint64_t i = 0; i < n_ext; ++i) {
        if (!(ext[i].flags & MKSNAP_X_CDC))
            continue;
        if (groups[i] >= st.n_groups)
            return fail(h, MKSNAP_E_INVAL, "group out of range");
        if ((ext[i].flags & MKSNAP_X_CONT) && h->file_open && groups[i] != st.open_group)
            return fail(h, MKSNAP_E_INVAL, "a continuation carries another group than its file");
    }
    // chunks per CDC extent, counted before the plain submit hands the arena back (a split file yields its chunks
    // with its last piece, like the engine)
    const uint8_t *a = h->arenas[arena_id].data();
    std::vector<uint8_t> open = st.open_bytes;
    std::vector<std::pair<uint32_t, size_t>> tags;
    uint32_t open_group = st.open_group;
    for (uint64_t i = 0; i < n_ext; ++i) {
        const mksnap_extent &e = ext[i];
        if (!(e.flags & MKSNAP_X_CDC) || e.arena_off + e.len > used)
            continue; // the plain submit rejects an out-of-bounds extent
        const bool cont = e.flags & MKSNAP_X_CONT, more = e.flags & MKSNAP_X_MORE;
        if (cont || more) {
            open.insert(open.end(), a + e.arena_off, a + e.arena_off + e.len);
            if (more) {
                open_group = groups[i];
                continue;
            }
            tags.emplace_back(groups[i], count_cuts(h, open.data(), open.size()));
            open.clear();
        } else {
            tags.emplace_back(groups[i], count_cuts(h, a + e.arena_off, e.len));
        }
    }
    const int rc = mock_plain_arena_submit(h, arena_id, used, ext, n_ext, rng, n_rng);
    if (rc)
        return rc;
    st.open_bytes.swap(open);
    st.open_group = open_group;
    for (const auto &t : tags)
        st.chunk_group.insert(st.chunk_group.end(), t.second, t.first);
    for (uint64_t i = 0; i < n_ext; ++i)
        if (ext[i].flags & MKSNAP_X_CDC) {
            st.res[groups[i]].cdc_bytes += ext[i].len;
            st.res[groups[i]].n_files += (ext[i].flags & MKSNAP_X_CONT) ? 0 : 1;
        }
    return 0;
}

int mksnap_finish(mksnap_t *h, mksnap_result *out)
{
    const int rc = mock_plain_finish(h, out);
    auto it = h && rc == 0 ? g_groups.find(h) : g_groups.end();
    if (it == g_groups.end())
        return rc;
    GroupState &st = it->second;
    if (st.chunk_group.size() * 32 != h->digests.size())
        return fail(h, MKSNAP_E_STATE, "internal: chunk groups disagree with the chunk count");
    uint64_t first_row = 0;
    for (uint32_t g = 0; g < st.n_groups; ++g) { // each group's table as if its chunks were a session of their own
        std::vector<uint8_t> t;
        for (size_t c = 0; c < st.chunk_group.size(); ++c)
            if (st.chunk_group[c] == g)
                t.insert(t.end(), h->digests.begin() + 32 * c, h->digests.begin() + 32 * c + 32);
        mksnap_group_result &r = st.res[g];
        r.n_chunks = t.size() / 32;
        r.n_unique = mko_sort_unique_digests(t.data(), t.size() / 32);
        r.first_row = first_row;
        first_row += r.n_unique;
        mko_merkle_root(t.data(), r.n_unique, r.root);
    }
    return 0;
}

int mksnap_get_group_results(mksnap_t *h, mksnap_group_result *out, uint32_t n_groups)
{
    if (!h || !out)
        return MKSNAP_E_INVAL;
    auto it = g_groups.find(h);
    if (it == g_groups.end() || !h->finished)
        return fail(h, MKSNAP_E_STATE, "get_group_results needs a finished grouped session");
    if (n_groups != it->second.n_groups)
        return fail(h, MKSNAP_E_INVAL, "n_groups differs from the session's");
    memcpy(out, it->second.res.data(), n_groups * sizeof *out);
    return 0;
}

} // extern "C"
