// vindex.cu — host-side mirror of the reference's IVectorIndex classes on top of the row-ordinal C ABI.
//
// Pure host code (no kernels): it owns what the C# classes own besides the vectors — the string ids, the
// id -> row dictionaries and the Add / Upsert / Delete / Build bookkeeping — and drives libpyrope_gpu's
// row-ordinal entry points for everything that touches a vector.  One pyrope_vindex stands for one of
//   BruteForceVectorIndex (Vector/BruteForceVectorIndex.cs)   kind FLAT
//   IvfFlatVectorIndex    (Vector/IvfFlatVectorIndex.cs)      kind IVF_FLAT
//   IvfPqVectorIndex      (Vector/IvfPqVectorIndex.cs)        kind IVF_PQ
//   DeltaVectorIndex      (Vector/DeltaVectorIndex.cs)        head + tail, both of the above
// Every row carries the process-wide ordinal of its id string as its LABEL, so a head and a tail that were
// created separately (as DeltaVectorIndexTests.cs and VectorIndexRegistry.cs:110-111 do) agree on identity and
// the Head+Tail merge can de-duplicate on the device.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../include/pyrope_gpu.h"
#include "internal.h"

namespace {

thread_local std::string g_verr;

int vfail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_verr = buf;
    return code;
}
// an error raised by the row-ordinal layer: keep its code, copy its message
int vpass(int rc) {
    if (rc != PYROPE_OK) g_verr = pyrope_last_error();
    return rc;
}
// the same for the sharded layer, which keeps its own message
int spass(int rc) {
    if (rc != PYROPE_OK) g_verr = pyrope_sharded_last_error();
    return rc;
}
#define VTRY(expr)                            \
    do {                                      \
        int _r = (expr);                      \
        if (_r != PYROPE_OK) return vpass(_r); \
    } while (0)
// a status whose message is already in g_verr
#define LTRY(expr)                       \
    do {                                 \
        int _r = (expr);                 \
        if (_r != PYROPE_OK) return _r;  \
    } while (0)

// process-wide id table: string -> ordinal (the row label), ordinal -> string.  Entries are reference counted — one
// reference per leaf index whose row_of holds the id — and an ordinal whose count drops to zero is recycled, so a
// long-lived server with id churn does not grow the table without bound.  (A caller turns search results into strings
// before it lets go of the index's read lock, as the reference's Search does by returning the strings themselves.)
struct IdEntry { std::string s; int64_t refs = 0; bool used = false; };
std::mutex g_id_mu;
std::vector<IdEntry> g_ids;
std::vector<int64_t> g_free_gids;
std::unordered_map<std::string, int64_t> g_gid_of;

// find or create; a fresh entry has no references yet (id_ref / id_drop_if_unreferenced follow)
int64_t intern_id(const std::string& id) {
    std::lock_guard<std::mutex> g(g_id_mu);
    auto it = g_gid_of.find(id);
    if (it != g_gid_of.end()) return it->second;
    int64_t gid;
    if (!g_free_gids.empty()) { gid = g_free_gids.back(); g_free_gids.pop_back(); }
    else { gid = (int64_t)g_ids.size(); g_ids.emplace_back(); }
    g_ids[(size_t)gid].s = id;
    g_ids[(size_t)gid].refs = 0;
    g_ids[(size_t)gid].used = true;
    g_gid_of.emplace(id, gid);
    return gid;
}
int64_t lookup_id(const std::string& id) {
    std::lock_guard<std::mutex> g(g_id_mu);
    auto it = g_gid_of.find(id);
    return it == g_gid_of.end() ? -1 : it->second;
}
void id_ref(int64_t gid) {
    std::lock_guard<std::mutex> g(g_id_mu);
    if (gid >= 0 && gid < (int64_t)g_ids.size() && g_ids[(size_t)gid].used) g_ids[(size_t)gid].refs++;
}
void id_release_locked(int64_t gid) {
    IdEntry& e = g_ids[(size_t)gid];
    g_gid_of.erase(e.s);
    e.s.clear();
    e.s.shrink_to_fit();
    e.used = false;
    e.refs = 0;
    g_free_gids.push_back(gid);
}
void id_unref(int64_t gid) {
    std::lock_guard<std::mutex> g(g_id_mu);
    if (gid < 0 || gid >= (int64_t)g_ids.size() || !g_ids[(size_t)gid].used) return;
    if (--g_ids[(size_t)gid].refs <= 0) id_release_locked(gid);
}
void id_drop_if_unreferenced(int64_t gid) {  // an Add that failed after interning a brand-new id
    std::lock_guard<std::mutex> g(g_id_mu);
    if (gid >= 0 && gid < (int64_t)g_ids.size() && g_ids[(size_t)gid].used && g_ids[(size_t)gid].refs <= 0) id_release_locked(gid);
}

bool blank(const char* id) {  // string.IsNullOrWhiteSpace
    if (!id) return true;
    for (const unsigned char* p = (const unsigned char*)id; *p; ++p)
        if (!isspace(*p)) return false;
    return true;
}

}  // namespace

struct pyrope_vindex {
    int kind = 0, dim = 0, metric = 0;
    pyrope_index* h = nullptr;      // one-device leaf (null for a delta)
    pyrope_sharded* sh = nullptr;   // or a leaf over several devices (pyrope_vindex_create_sharded)
    // delta
    pyrope_vindex* head = nullptr;
    pyrope_vindex* tail = nullptr;
    pyrope_delta* d = nullptr;
    std::shared_mutex lock;  // ReaderWriterLockSlim of the reference classes
    // id bookkeeping of one leaf index
    std::unordered_map<int64_t, int64_t> row_of;     // gid -> row ordinal currently answering for the id
    std::unordered_set<int64_t> buffered;            // IVF: gids whose current row sits in the write buffer
    std::unordered_map<int64_t, int64_t> shadowed;   // IVF: gid -> list row hidden behind its buffered copy
    std::vector<int64_t> gid_of_row;                 // row ordinal -> gid (-1 once the row is gone)
    bool built = false;

    void note_row(int64_t row, int64_t gid) {
        if ((int64_t)gid_of_row.size() <= row) gid_of_row.resize((size_t)row + 1, -1);
        gid_of_row[(size_t)row] = gid;
    }
    // row_of owns one reference per id it holds
    void set_row(int64_t gid, int64_t row) {
        auto it = row_of.find(gid);
        if (it == row_of.end()) { row_of.emplace(gid, row); id_ref(gid); }
        else it->second = row;
    }
    std::unordered_map<int64_t, int64_t>::iterator drop(std::unordered_map<int64_t, int64_t>::iterator it) {
        const int64_t gid = it->first;
        auto nx = row_of.erase(it);
        id_unref(gid);
        return nx;
    }
    void drop_all() {
        for (auto& kv : row_of) id_unref(kv.first);
        row_of.clear();
    }
};

namespace {

typedef pyrope_vindex V;

int check_vec(const V* v, const float* vec, int len) {
    if (!vec) return vfail(PYROPE_ERR_INVALID_ARG, "Value cannot be null. (Parameter 'vector')");
    if (len != v->dim) return vfail(PYROPE_ERR_DIMENSION, "Vector dimension mismatch");
    return PYROPE_OK;
}

// ---- the row-ordinal handle behind a leaf: one device (pyrope_index_*) or several (pyrope_sharded_*).  Errors come
// back with their message in g_verr.
int row_add(V* v, int64_t gid, const float* vec, int64_t* row) {
    return v->sh ? spass(pyrope_sharded_add_batch(v->sh, 1, vec, &gid, row)) : vpass(pyrope_index_add_batch(v->h, 1, vec, &gid, row));
}
int row_update(V* v, int64_t row, const float* vec) {
    return v->sh ? spass(pyrope_sharded_update_row(v->sh, row, vec)) : vpass(pyrope_index_update_row(v->h, row, vec));
}
int row_shadow(V* v, int64_t row, int shadowed) {
    return v->sh ? spass(pyrope_sharded_shadow_row(v->sh, row, shadowed)) : vpass(pyrope_index_shadow_row(v->h, row, shadowed));
}
int row_delete(V* v, int64_t row) {
    return v->sh ? spass(pyrope_sharded_delete_row(v->sh, row)) : vpass(pyrope_index_delete_row(v->h, row));
}
int row_build(V* v) { return v->sh ? spass(pyrope_sharded_build(v->sh)) : vpass(pyrope_index_build(v->h)); }
int row_extend(V* v) { return v->sh ? spass(pyrope_sharded_extend(v->sh)) : vpass(pyrope_index_extend(v->h)); }
int row_is_built(V* v, int* out) { return v->sh ? spass(pyrope_sharded_is_built(v->sh, out)) : vpass(pyrope_index_is_built(v->h, out)); }
int row_set_labels(V* v, int64_t n, const int64_t* labels) {
    return v->sh ? spass(pyrope_sharded_set_labels(v->sh, n, labels)) : vpass(pyrope_index_set_labels(v->h, n, labels));
}
int row_snapshot(V* v, const char* path) {
    return v->sh ? spass(pyrope_sharded_snapshot(v->sh, path)) : vpass(pyrope_index_snapshot(v->h, path));
}
int row_load(V* v, const char* path) { return v->sh ? spass(pyrope_sharded_load(v->sh, path)) : vpass(pyrope_index_load(v->h, path)); }
int row_snapshot_next_row(V* v, const char* path, int64_t* next_row) {
    return v->sh ? spass(pyrope_internal_sharded_snapshot_next_row(path, next_row))
                 : vpass(pyrope_internal_snapshot_next_row(path, next_row));
}

// ---- leaf writes (no locking; callers hold the write lock) ------------------------------------------------
int leaf_add_new(V* v, int64_t gid, const float* vec) {
    int64_t row = -1;
    LTRY(row_add(v, gid, vec, &row));
    v->set_row(gid, row);
    v->note_row(row, gid);
    if (v->kind != PYROPE_FLAT) v->buffered.insert(gid);
    return PYROPE_OK;
}

// IVF: `_buffer[id] = entry` (IvfFlatVectorIndex.cs:47, IvfPqVectorIndex.cs:42)
int leaf_buffer_set(V* v, int64_t gid, const float* vec) {
    auto it = v->row_of.find(gid);
    if (it == v->row_of.end()) return leaf_add_new(v, gid, vec);
    if (v->buffered.count(gid)) return row_update(v, it->second, vec);  // key keeps its slot
    // the id sits in an inverted list: the buffered copy shadows it (seenIds, IvfFlatVectorIndex.cs:210,
    // IvfPqVectorIndex.cs:170) until the next Build
    const int64_t old = it->second;
    LTRY(row_shadow(v, old, 1));
    v->shadowed[gid] = old;
    return leaf_add_new(v, gid, vec);
}

int leaf_add(V* v, const char* id, const float* vec, int len, bool upsert) {
    if (v->kind != PYROPE_IVF_PQ && blank(id))  // IvfPqVectorIndex.Add validates nothing (:36-45)
        return vfail(PYROPE_ERR_INVALID_ARG, v->kind == PYROPE_FLAT ? "Id cannot be empty. (Parameter 'id')" : "Id empty");
    if (!id) return vfail(PYROPE_ERR_INVALID_ARG, "Value cannot be null. (Parameter 'key')");
    int r = check_vec(v, vec, len);  // IVF_PQ stores any array and fails at Build; the device copy cannot
    if (r != PYROPE_OK) return r;
    const int64_t gid = intern_id(id);
    int rc;
    if (v->kind != PYROPE_FLAT) rc = leaf_buffer_set(v, gid, vec);
    else {
        auto it = v->row_of.find(gid);
        if (it == v->row_of.end()) rc = leaf_add_new(v, gid, vec);
        else if (!upsert)  // BruteForceVectorIndex.cs:141-144
            rc = vfail(PYROPE_ERR_INVALID_STATE, "Vector with id '%s' already exists.", id);
        else rc = row_update(v, it->second, vec);  // :203-206 in place, scan position kept
    }
    if (rc != PYROPE_OK) id_drop_if_unreferenced(gid);
    return rc;
}

int leaf_delete(V* v, const char* id, bool* removed) {
    *removed = false;
    if (v->kind != PYROPE_IVF_PQ && blank(id))
        return vfail(PYROPE_ERR_INVALID_ARG, v->kind == PYROPE_FLAT ? "Id cannot be empty. (Parameter 'id')" : "Id empty");
    if (!id) return vfail(PYROPE_ERR_INVALID_ARG, "Value cannot be null. (Parameter 'key')");
    const int64_t gid = lookup_id(id);
    if (gid < 0) return PYROPE_OK;
    auto it = v->row_of.find(gid);
    if (it == v->row_of.end()) return PYROPE_OK;
    const int64_t row = it->second;
    if (v->kind == PYROPE_FLAT) {  // BruteForceVectorIndex.cs:231-254: tombstone, id leaves the map
        LTRY(row_delete(v, row));
        v->gid_of_row[(size_t)row] = -1;
        v->drop(it);
        *removed = true;
        return PYROPE_OK;
    }
    const bool in_buffer = v->buffered.count(gid) != 0;
    if (v->kind == PYROPE_IVF_PQ) {  // IvfPqVectorIndex.cs:48-53: only the buffer
        if (!in_buffer) return PYROPE_OK;
        LTRY(row_delete(v, row));
        v->gid_of_row[(size_t)row] = -1;
        v->buffered.erase(gid);
        auto sh = v->shadowed.find(gid);
        if (sh != v->shadowed.end()) {  // the encoded copy is visible again
            LTRY(row_shadow(v, sh->second, 0));
            it->second = sh->second;
            v->shadowed.erase(sh);
        } else {
            v->drop(it);
        }
        *removed = true;
        return PYROPE_OK;
    }
    // IvfFlatVectorIndex.cs:62-83: buffer entry and every list entry with this id
    LTRY(row_delete(v, row));
    v->gid_of_row[(size_t)row] = -1;
    auto sh = v->shadowed.find(gid);
    if (sh != v->shadowed.end()) {
        LTRY(row_delete(v, sh->second));
        v->gid_of_row[(size_t)sh->second] = -1;
        v->shadowed.erase(sh);
    }
    v->buffered.erase(gid);
    v->drop(it);
    *removed = true;
    return PYROPE_OK;
}

// bookkeeping of a finished Build
void leaf_after_build(V* v, bool had_buffer) {
    if (v->kind == PYROPE_FLAT) return;
    if (v->kind == PYROPE_IVF_PQ) {
        if (!had_buffer) return;  // IvfPqVectorIndex.cs:62-65: nothing buffered, nothing changes
        // :92-109: the lists are REPLACED by the buffer's rows; ids that were only encoded are gone
        for (auto it = v->row_of.begin(); it != v->row_of.end();) {
            if (!v->buffered.count(it->first)) {
                v->gid_of_row[(size_t)it->second] = -1;
                it = v->drop(it);
            } else {
                ++it;
            }
        }
    }
    for (auto& kv : v->shadowed) v->gid_of_row[(size_t)kv.second] = -1;  // replaced by the buffered copy
    v->shadowed.clear();
    v->buffered.clear();
    if (!v->row_of.empty()) v->built = true;
}

int leaf_build(V* v) {
    if (v->kind == PYROPE_FLAT) return PYROPE_OK;
    const bool had_buffer = !v->buffered.empty();
    LTRY(row_build(v));
    leaf_after_build(v, had_buffer);
    return PYROPE_OK;
}

// bookkeeping of a finished Extend: the buffered ids are now list ids under the same row ordinals, the list rows they
// shadowed are deleted.  Unlike an IVF_PQ Build, no id that was only encoded is dropped.
void leaf_after_extend(V* v) {
    for (auto& kv : v->shadowed) v->gid_of_row[(size_t)kv.second] = -1;
    v->shadowed.clear();
    v->buffered.clear();
    if (!v->row_of.empty()) v->built = true;
}

int leaf_extend(V* v) {
    LTRY(row_extend(v));  // FLAT -> UNSUPPORTED, not built -> INVALID_STATE
    leaf_after_extend(v);
    return PYROPE_OK;
}

// DeltaVectorIndex.Build's move (:133-147): the head's live rows go to the tail's buffer, the id tables follow them.
// Caller holds the unique locks of the delta and both sides.
int delta_move_with_ids(V* v) {
    V* hd = v->head;
    V* tl = v->tail;
    std::vector<int64_t> moved_gids;  // head scan order = row order, live rows only
    for (size_t r = 0; r < hd->gid_of_row.size(); ++r)
        if (hd->gid_of_row[r] >= 0) moved_gids.push_back(hd->gid_of_row[r]);
    std::vector<int64_t> tail_rows(moved_gids.size() + 1, -1);
    int64_t moved = 0;
    VTRY(pyrope_delta_move(v->d, &moved, tail_rows.data()));
    if (moved != (int64_t)moved_gids.size())
        return vfail(PYROPE_ERR_INVALID_STATE, "compaction moved %lld rows, the id table expected %zu", (long long)moved,
                     moved_gids.size());
    for (size_t i = 0; i < moved_gids.size(); ++i) {  // what _tail.Add(id, vec) does to the tail's tables
        const int64_t gid = moved_gids[i], row = tail_rows[i];
        auto it = tl->row_of.find(gid);
        if (it != tl->row_of.end() && !tl->buffered.count(gid) && it->second != row) tl->shadowed[gid] = it->second;
        tl->set_row(gid, row);
        tl->note_row(row, gid);
        if (tl->kind != PYROPE_FLAT) tl->buffered.insert(gid);
    }
    std::fill(hd->gid_of_row.begin(), hd->gid_of_row.end(), (int64_t)-1);  // _head.Delete(id) for every moved id
    hd->drop_all();
    return PYROPE_OK;
}

int64_t leaf_count(const V* v) {
    if (v->kind == PYROPE_IVF_PQ) return 0;  // IvfPqVectorIndex.cs:230 hard-codes 0
    // IvfFlatVectorIndex.cs:300-312 counts buffer entries plus every list entry, shadowed ones included
    return (int64_t)v->row_of.size() + (int64_t)v->shadowed.size();
}

// ---- file helpers for the id table ------------------------------------------------------------------------
bool put64(FILE* f, int64_t x) { return fwrite(&x, 8, 1, f) == 1; }
bool get64(FILE* f, int64_t* x) { return fread(x, 8, 1, f) == 1; }

// id table of one leaf: every live row (ordinal, id string) + which ids are buffered / shadowed
int leaf_save_ids(const V* v, const std::string& path) {
    const std::string tmp = path + ".tmp";
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) return vfail(PYROPE_ERR_INVALID_ARG, "cannot open %s for writing", tmp.c_str());
    bool ok = put64(f, 0x5044495650ll) && put64(f, (int64_t)v->gid_of_row.size()) && put64(f, v->built ? 1 : 0);
    int64_t live = 0;
    for (int64_t g : v->gid_of_row) live += g >= 0;
    ok = ok && put64(f, live);
    {
        std::lock_guard<std::mutex> g(g_id_mu);
        for (size_t r = 0; ok && r < v->gid_of_row.size(); ++r) {
            const int64_t gid = v->gid_of_row[r];
            if (gid < 0) continue;
            const std::string& s = g_ids[(size_t)gid].s;
            int64_t state = 0;  // 0 current row (list or FLAT), 1 current row in the buffer, 2 shadowed list row
            auto ro = v->row_of.find(gid);
            if (ro != v->row_of.end() && ro->second == (int64_t)r) state = v->buffered.count(gid) ? 1 : 0;
            else state = 2;
            ok = put64(f, (int64_t)r) && put64(f, state) && put64(f, (int64_t)s.size()) &&
                 (s.empty() || fwrite(s.data(), 1, s.size(), f) == s.size());
        }
    }
    if (fclose(f) != 0 || !ok) { remove(tmp.c_str()); return vfail(PYROPE_ERR_INVALID_ARG, "short write to %s", tmp.c_str()); }
    if (rename(tmp.c_str(), path.c_str()) != 0) { remove(tmp.c_str()); return vfail(PYROPE_ERR_INVALID_ARG, "cannot move %s into place", tmp.c_str()); }
    return PYROPE_OK;
}

// The id table of a snapshot, parsed and validated on its own: pyrope_vindex_load reads it BEFORE the index file is
// loaded and applies it after, so a missing or corrupt table never leaves freshly loaded rows under foreign labels.
struct LoadedIds {
    int64_t nrows = 0, built = 0;
    std::vector<std::pair<int64_t, std::string>> rows;  // (row ordinal, id)
    std::vector<int64_t> state;                         // 0 current, 1 current + buffered, 2 shadowed list row
};
int leaf_parse_ids(const std::string& path, LoadedIds& L) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return vfail(PYROPE_ERR_NOT_FOUND, "Snapshot file not found. (%s)", path.c_str());
    int64_t magic = 0, live = 0;
    bool ok = get64(f, &magic) && magic == 0x5044495650ll && get64(f, &L.nrows) && get64(f, &L.built) && get64(f, &live) &&
              L.nrows >= 0 && live >= 0 && live <= L.nrows;
    std::vector<uint8_t> seen((size_t)(ok ? L.nrows : 0), 0);
    std::string s;
    for (int64_t i = 0; ok && i < live; ++i) {
        int64_t r = 0, state = 0, len = 0;
        ok = get64(f, &r) && get64(f, &state) && get64(f, &len) && r >= 0 && r < L.nrows && !seen[(size_t)r] && state >= 0 &&
             state <= 2 && len >= 0 && len < (1 << 20);
        if (!ok) break;
        seen[(size_t)r] = 1;
        s.resize((size_t)len);
        ok = len == 0 || fread(&s[0], 1, (size_t)len, f) == (size_t)len;
        if (!ok) break;
        L.rows.emplace_back(r, s);
        L.state.push_back(state);
    }
    fclose(f);
    if (!ok) return vfail(PYROPE_ERR_INVALID_ARG, "%s is not a pyrope id table", path.c_str());
    return PYROPE_OK;
}
int leaf_apply_ids(V* v, const LoadedIds& L) {
    std::vector<int64_t> gid_of_row((size_t)L.nrows, -1);
    std::unordered_map<int64_t, int64_t> row_of, shadowed;
    std::unordered_set<int64_t> buffered;
    for (size_t i = 0; i < L.rows.size(); ++i) {
        const int64_t r = L.rows[i].first, gid = intern_id(L.rows[i].second);
        gid_of_row[(size_t)r] = gid;
        if (L.state[i] == 2) shadowed[gid] = r;
        else {
            if (row_of.emplace(gid, r).second) id_ref(gid);
            else row_of[gid] = r;
            if (L.state[i] == 1) buffered.insert(gid);
        }
    }
    for (auto& kv : shadowed)  // a shadowed row without its buffered copy cannot be written by leaf_save_ids; keep the id alive anyway
        if (!row_of.count(kv.first)) { row_of.emplace(kv.first, kv.second); id_ref(kv.first); }
    // the rows in the library's snapshot carry the labels of the process that wrote it: re-label them.  Rows that are
    // gone get -1, which no search returns and no live id ordinal equals.
    int rc = row_set_labels(v, L.nrows, gid_of_row.data());
    if (rc != PYROPE_OK) {
        for (auto& kv : row_of) id_unref(kv.first);
        return rc;
    }
    v->drop_all();
    v->gid_of_row.swap(gid_of_row);
    v->row_of.swap(row_of);
    v->shadowed.swap(shadowed);
    v->buffered.swap(buffered);
    v->built = L.built != 0;
    return PYROPE_OK;
}
// index file + id table of one leaf, all or nothing as far as validation goes
int leaf_load(V* v, const std::string& path) {
    LoadedIds L;
    int r = leaf_parse_ids(path + ".ids", L);
    if (r != PYROPE_OK) return r;
    int64_t next_row = -1;
    LTRY(row_snapshot_next_row(v, path.c_str(), &next_row));
    if (L.nrows < next_row)
        return vfail(PYROPE_ERR_INVALID_ARG, "%s.ids covers %lld rows, the snapshot holds %lld", path.c_str(), (long long)L.nrows,
                     (long long)next_row);
    LTRY(row_load(v, path.c_str()));
    return leaf_apply_ids(v, L);
}

}  // namespace

extern "C" {

const char* pyrope_vindex_last_error(void) { return g_verr.c_str(); }

int pyrope_vindex_create(int kind, int dim, int metric, int nlist, int pq_m, int pq_k, pyrope_vindex** out) {
    if (!out) return vfail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    V* v = new (std::nothrow) V();
    if (!v) return vfail(PYROPE_ERR_OOM, "out of host memory");
    int rc = pyrope_index_create(kind, dim, metric, nlist, pq_m, pq_k, &v->h);
    if (rc != PYROPE_OK) {
        delete v;
        return vpass(rc);
    }
    v->kind = kind; v->dim = dim; v->metric = metric;
    *out = v;
    return PYROPE_OK;
}

int pyrope_vindex_create_sharded(int n_devices, const int* devices, int kind, int dim, int metric, int nlist, int pq_m, int pq_k,
                                 pyrope_vindex** out) {
    if (!out) return vfail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (kind != PYROPE_IVF_FLAT && kind != PYROPE_IVF_PQ) return vfail(PYROPE_ERR_UNSUPPORTED, "a sharded index must be IVF_FLAT or IVF_PQ");
    V* v = new (std::nothrow) V();
    if (!v) return vfail(PYROPE_ERR_OOM, "out of host memory");
    int rc = pyrope_sharded_create(n_devices, devices, kind, dim, metric, nlist, pq_m, pq_k, &v->sh);
    if (rc != PYROPE_OK) {
        delete v;
        return spass(rc);
    }
    v->kind = kind; v->dim = dim; v->metric = metric;
    *out = v;
    return PYROPE_OK;
}

int pyrope_vindex_create_delta(pyrope_vindex* head, pyrope_vindex* tail, pyrope_vindex** out) {
    if (!out) return vfail(PYROPE_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (!head || !tail || head->d || tail->d) return vfail(PYROPE_ERR_INVALID_ARG, "head and tail must be leaf indexes");
    if (head->sh) return vfail(PYROPE_ERR_UNSUPPORTED, "the head must be a one-device FLAT index");
    V* v = new (std::nothrow) V();
    if (!v) return vfail(PYROPE_ERR_OOM, "out of host memory");
    int rc = tail->sh ? pyrope_delta_create_sharded(head->h, tail->sh, &v->d)  // DeltaVectorIndex..ctor :18-28
                      : pyrope_delta_create(head->h, tail->h, &v->d);
    if (rc != PYROPE_OK) {
        delete v;
        return vpass(rc);
    }
    v->kind = -1; v->dim = head->dim; v->metric = head->metric;
    v->head = head; v->tail = tail;
    *out = v;
    return PYROPE_OK;
}

int pyrope_vindex_destroy(pyrope_vindex* v) {
    if (!v) return PYROPE_OK;
    if (v->d) pyrope_delta_destroy(v->d);  // the two sides stay alive: they were only borrowed
    if (v->h) pyrope_index_destroy(v->h);
    if (v->sh) pyrope_sharded_destroy(v->sh);
    v->drop_all();
    delete v;
    return PYROPE_OK;
}

int pyrope_vindex_native(pyrope_vindex* v, pyrope_index** out) {
    if (!v || !out) return vfail(PYROPE_ERR_INVALID_ARG, "null argument");
    *out = v->h;
    return PYROPE_OK;
}

int pyrope_vindex_set_quantization(pyrope_vindex* v, int enable) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (v->d || v->kind != PYROPE_FLAT) return vfail(PYROPE_ERR_INVALID_STATE, "EnableQuantization exists on BruteForceVectorIndex only");
    std::unique_lock<std::shared_mutex> g(v->lock);
    return vpass(pyrope_index_set_quantization(v->h, enable));
}

int pyrope_vindex_add(pyrope_vindex* v, const char* id, const float* vec, int len) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::unique_lock<std::shared_mutex> g(v->lock);
    if (!v->d) return leaf_add(v, id, vec, len, false);
    std::unique_lock<std::shared_mutex> gh(v->head->lock);
    return leaf_add(v->head, id, vec, len, false);  // DeltaVectorIndex.cs:30-44: writes go to the head
}

int pyrope_vindex_upsert(pyrope_vindex* v, const char* id, const float* vec, int len) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::unique_lock<std::shared_mutex> g(v->lock);
    if (!v->d) return leaf_add(v, id, vec, len, true);
    std::unique_lock<std::shared_mutex> gh(v->head->lock);
    return leaf_add(v->head, id, vec, len, true);  // :46-57
}

int pyrope_vindex_delete(pyrope_vindex* v, const char* id, int* removed_out) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (removed_out) *removed_out = 0;
    std::unique_lock<std::shared_mutex> g(v->lock);
    bool a = false, b = false;
    if (!v->d) {
        int r = leaf_delete(v, id, &a);
        if (r != PYROPE_OK) return r;
    } else {  // :59-74: both sides, h || t
        std::unique_lock<std::shared_mutex> gh(v->head->lock);
        std::unique_lock<std::shared_mutex> gt(v->tail->lock);
        int r = leaf_delete(v->head, id, &a);
        if (r != PYROPE_OK) return r;
        r = leaf_delete(v->tail, id, &b);
        if (r != PYROPE_OK) return r;
    }
    if (removed_out) *removed_out = (a || b) ? 1 : 0;
    return PYROPE_OK;
}

int pyrope_vindex_build(pyrope_vindex* v) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::unique_lock<std::shared_mutex> g(v->lock);
    if (!v->d) return leaf_build(v);
    // DeltaVectorIndex.Build :124-158 — compaction: head rows move to the tail device-to-device
    V* hd = v->head;
    V* tl = v->tail;
    std::unique_lock<std::shared_mutex> gh(hd->lock);
    std::unique_lock<std::shared_mutex> gt(tl->lock);
    const bool had_buffer = !tl->buffered.empty() || !hd->row_of.empty();
    // move first, book-keeping second, the tail's Build last: if the build fails (out of memory in k-means, say) the id
    // tables already describe where every row is, so Delete / Upsert / Snapshot keep working and Build can be retried
    LTRY(delta_move_with_ids(v));
    VTRY(pyrope_delta_build_tail(v->d));
    leaf_after_build(tl, had_buffer);
    return PYROPE_OK;
}

int pyrope_vindex_extend(pyrope_vindex* v) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::unique_lock<std::shared_mutex> g(v->lock);
    if (!v->d) return leaf_extend(v);
    // compaction by Extend: the move of pyrope_vindex_build, then the tail's Extend instead of its Build
    V* hd = v->head;
    V* tl = v->tail;
    std::unique_lock<std::shared_mutex> gh(hd->lock);
    std::unique_lock<std::shared_mutex> gt(tl->lock);
    // a tail that cannot be extended refuses before any row moves
    if (tl->kind == PYROPE_FLAT) return vfail(PYROPE_ERR_UNSUPPORTED, "Extend needs an IVF tail: FLAT has no inverted lists");
    int built = 0;
    LTRY(row_is_built(tl, &built));
    if (!built) return vfail(PYROPE_ERR_INVALID_STATE, "Extend needs a built tail: call Build first");
    LTRY(delta_move_with_ids(v));
    VTRY(pyrope_delta_extend_tail(v->d));
    leaf_after_extend(tl);
    return PYROPE_OK;
}

int pyrope_vindex_search(pyrope_vindex* v, int64_t nq, const float* Q, int len, int topk, int64_t max_scans, int nprobe,
                         float* scores_out, int64_t* gids_out, int32_t* counts_out) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    const int kind = v->d ? (int)PYROPE_FLAT : v->kind;  // a delta validates like its FLAT head, which runs first
    if (kind != PYROPE_IVF_PQ) {                          // IvfPqVectorIndex.Search validates nothing (:118-125)
        int r = check_vec(v, Q, len);
        if (r != PYROPE_OK) return r;
    } else if (!Q || len != v->dim) {
        return vfail(PYROPE_ERR_DIMENSION, "Vector dimension mismatch");
    }
    std::shared_lock<std::shared_mutex> g(v->lock);
    if (v->d) return vpass(pyrope_delta_search_batch(v->d, nq, Q, topk, max_scans, nprobe, scores_out, gids_out, counts_out));
    if (v->sh) return spass(pyrope_sharded_search_batch(v->sh, nq, Q, topk, max_scans, nprobe, scores_out, gids_out, counts_out));
    return vpass(pyrope_index_search_batch(v->h, nq, Q, topk, max_scans, nprobe, scores_out, gids_out, counts_out));
}

// csrc/batcher.cu (internal): what a Search with topK <= 0 or a large topK gives on this index, so the batcher can answer
// such a caller alone.  max_topk: the largest topK Search accepts; nonpos_empty: topK <= 0 returns an empty result
// (an IVF leaf) rather than OUT_OF_RANGE (a FLAT leaf, or a delta whose FLAT head validates first).
int pyrope_internal_vindex_limits(pyrope_vindex* v, int* dim_out, int* max_topk_out, int* nonpos_empty_out) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    int lim = 1024, empty = 0;
    if (v->d) {
        VTRY(pyrope_internal_delta_limits(v->d, nullptr, &lim));
    } else if (v->sh) {
        int n = 1;
        LTRY(spass(pyrope_sharded_device_count(v->sh, &n)));
        lim = std::min(1024, 4096 / n);  // pyrope_sharded_search_batch: n x topK candidates in one merge
        empty = 1;
    } else {
        empty = v->kind != PYROPE_FLAT;
    }
    if (dim_out) *dim_out = v->dim;
    if (max_topk_out) *max_topk_out = lim;
    if (nonpos_empty_out) *nonpos_empty_out = empty;
    return PYROPE_OK;
}

// csrc/batcher.cu (internal): one batched Search under the shared lock, as pyrope_vindex_search runs it, with query i
// asking for topks[i] (each in 1 .. the limit above).  Outputs have stride max(topks).  A delta merges with the per-query
// k (pyrope_delta_search_batch_topk); a leaf searches at max(topks), whose first topks[i] entries per query are that
// query's own top topks[i] — the caller keeps those.
int pyrope_internal_vindex_search_topk(pyrope_vindex* v, int64_t nq, const float* Q, const int32_t* topks, int64_t max_scans,
                                       int nprobe, float* scores_out, int64_t* gids_out, int32_t* counts_out) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (nq > 0 && (!Q || !topks)) return vfail(PYROPE_ERR_INVALID_ARG, "null argument");
    std::shared_lock<std::shared_mutex> g(v->lock);
    if (v->d) return vpass(pyrope_delta_search_batch_topk(v->d, nq, Q, topks, max_scans, nprobe, scores_out, gids_out, counts_out));
    int kmax = 1;
    for (int64_t i = 0; i < nq; ++i) kmax = std::max(kmax, (int)topks[i]);
    if (v->sh) return spass(pyrope_sharded_search_batch(v->sh, nq, Q, kmax, max_scans, nprobe, scores_out, gids_out, counts_out));
    return vpass(pyrope_index_search_batch(v->h, nq, Q, kmax, max_scans, nprobe, scores_out, gids_out, counts_out));
}

int pyrope_vindex_id(int64_t gid, char* buf, int cap, int* len_out) {
    std::lock_guard<std::mutex> g(g_id_mu);
    if (gid < 0 || gid >= (int64_t)g_ids.size() || !g_ids[(size_t)gid].used)
        return vfail(PYROPE_ERR_NOT_FOUND, "unknown id ordinal %lld", (long long)gid);
    const std::string& s = g_ids[(size_t)gid].s;
    if (len_out) *len_out = (int)s.size();
    if (buf && cap > 0) {
        const size_t n = std::min<size_t>(s.size(), (size_t)cap - 1);
        memcpy(buf, s.data(), n);
        buf[n] = 0;
    }
    return PYROPE_OK;
}

int pyrope_vindex_ids(const int64_t* gids, int64_t n, char* buf, int64_t cap, int64_t* offsets_out, int64_t* bytes_out) {
    if (n < 0 || (n > 0 && (!gids || !offsets_out))) return vfail(PYROPE_ERR_INVALID_ARG, "null argument");
    std::lock_guard<std::mutex> g(g_id_mu);  // one lock for the whole result list
    int64_t o = 0;
    for (int64_t i = 0; i < n; ++i) {
        offsets_out[i] = o;
        const int64_t gid = gids[i];
        if (gid < 0) continue;  // an empty result slot: zero-length string
        if (gid >= (int64_t)g_ids.size() || !g_ids[(size_t)gid].used)
            return vfail(PYROPE_ERR_NOT_FOUND, "unknown id ordinal %lld", (long long)gid);
        const std::string& s = g_ids[(size_t)gid].s;
        if (buf && o + (int64_t)s.size() <= cap) memcpy(buf + o, s.data(), s.size());
        o += (int64_t)s.size();
    }
    offsets_out[n] = o;
    if (bytes_out) *bytes_out = o;
    return PYROPE_OK;
}

int pyrope_vindex_id_table_size(int64_t* live_out, int64_t* slots_out) {
    std::lock_guard<std::mutex> g(g_id_mu);
    if (live_out) *live_out = (int64_t)g_gid_of.size();
    if (slots_out) *slots_out = (int64_t)g_ids.size();
    return PYROPE_OK;
}

int pyrope_vindex_stats(pyrope_vindex* v, int64_t* count_out, int* dim_out, int* metric_out) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    std::shared_lock<std::shared_mutex> g(v->lock);
    if (count_out) *count_out = v->d ? leaf_count(v->head) + leaf_count(v->tail) : leaf_count(v);  // DeltaVectorIndex.cs:232-236
    if (dim_out) *dim_out = v->dim;
    if (metric_out) *metric_out = v->metric;
    return PYROPE_OK;
}

int pyrope_vindex_get_centroids(pyrope_vindex* v, float* centroids_out, int* n_out) {
    if (!v || !n_out) return vfail(PYROPE_ERR_INVALID_ARG, "null argument");
    std::shared_lock<std::shared_mutex> g(v->lock);
    V* leaf = v->d ? v->tail : v;  // DeltaVectorIndex.cs:241-252: the tail's, if it has any
    *n_out = 0;
    if (leaf->kind == PYROPE_FLAT) return PYROPE_OK;  // not an ICentroidsProvider -> null
    if (leaf->sh) return spass(pyrope_sharded_get_centroids(leaf->sh, centroids_out, n_out));
    return vpass(pyrope_index_get_centroids(leaf->h, centroids_out, n_out));
}

int pyrope_vindex_snapshot(pyrope_vindex* v, const char* path) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (blank(path)) return vfail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty. (Parameter 'path')");  // BruteForceVectorIndex.cs:60
    std::shared_lock<std::shared_mutex> g(v->lock);
    const std::string base(path);
    if (!v->d) {
        LTRY(row_snapshot(v, path));
        return leaf_save_ids(v, base + ".ids");
    }
    VTRY(pyrope_delta_snapshot(v->d, path));
    int r = leaf_save_ids(v->head, base + ".head.ids");
    if (r != PYROPE_OK) return r;
    return leaf_save_ids(v->tail, base + ".tail.ids");
}

int pyrope_vindex_load(pyrope_vindex* v, const char* path) {
    if (!v) return vfail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (blank(path)) return vfail(PYROPE_ERR_INVALID_ARG, "Path cannot be empty. (Parameter 'path')");
    std::unique_lock<std::shared_mutex> g(v->lock);
    const std::string base(path);
    if (!v->d) return leaf_load(v, base);
    for (int side = 0; side < 2; ++side) {  // DeltaVectorIndex.cs:200-216: each side only if its file exists
        V* leaf = side == 0 ? v->head : v->tail;
        const std::string p = base + (side == 0 ? ".head" : ".tail");
        FILE* f = fopen(p.c_str(), "rb");
        if (!f) continue;
        fclose(f);
        int r = leaf_load(leaf, p);
        if (r != PYROPE_OK) return r;
    }
    return PYROPE_OK;
}

}  // extern "C"
