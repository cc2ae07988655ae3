// formats.cu — the data formats either side of the scan path (SURVEY §8f rank 4), host code only:
//   * VEC.ADD / VEC.SEARCH vector payloads: Utils/VectorParsing.cs:10-101 (JSON array, CSV / blank separated text,
//     raw little-endian float32 — the benchmark client's fast path, Benchmarks/Encoding/VectorEncoding.cs:8-16);
//   * FAISS-style *.fvecs datasets: Benchmarks/Datasets/FvecsReader.cs:14-60, plus a loader that streams a file
//     straight into an index's device storage.
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/pyrope_gpu.h"
#include "internal.h"

namespace {

// char.IsWhiteSpace restricted to what a single UTF-8 byte can encode
inline bool ws(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13); }
inline bool digit(unsigned char c) { return c >= '0' && c <= '9'; }

bool all_white(const unsigned char* p, int64_t n) {
    for (int64_t i = 0; i < n; ++i)
        if (!ws(p[i])) return false;
    return true;
}

// strtof on a validated, bounded token
float to_float(const unsigned char* p, int64_t n) {
    char small[64];
    std::string big;
    const char* s;
    if (n < (int64_t)sizeof small) {
        memcpy(small, p, (size_t)n);
        small[n] = 0;
        s = small;
    } else {
        big.assign((const char*)p, (size_t)n);
        s = big.c_str();
    }
    return strtof(s, nullptr);
}

// JSON number grammar (RFC 8259): -?(0|[1-9][0-9]*)(\.[0-9]+)?([eE][+-]?[0-9]+)?   -> chars consumed, 0 = no match
int64_t json_number(const unsigned char* p, int64_t n) {
    int64_t i = 0;
    if (i < n && p[i] == '-') ++i;
    if (i >= n) return 0;
    if (p[i] == '0') ++i;
    else if (p[i] >= '1' && p[i] <= '9') { while (i < n && digit(p[i])) ++i; }
    else return 0;
    if (i < n && p[i] == '.') {
        ++i;
        if (i >= n || !digit(p[i])) return 0;
        while (i < n && digit(p[i])) ++i;
    }
    if (i < n && (p[i] == 'e' || p[i] == 'E')) {
        ++i;
        if (i < n && (p[i] == '+' || p[i] == '-')) ++i;
        if (i >= n || !digit(p[i])) return 0;
        while (i < n && digit(p[i])) ++i;
    }
    return i;
}

// TryParseJsonVector (VectorParsing.cs:37-61): text[0] == '[' and JsonSerializer.Deserialize<float[]> succeeds with
// at least one element.  1 = parsed, 0 = not JSON (fall through), -1 = a number float cannot hold (Deserialize
// throws FormatException, which ParseVector does not catch).
int parse_json(const unsigned char* p, int64_t n, std::vector<float>& out) {
    if (n == 0 || p[0] != '[') return 0;
    auto skip = [&](int64_t& i) { while (i < n && (p[i] == ' ' || p[i] == '\t' || p[i] == '\n' || p[i] == '\r')) ++i; };
    int64_t i = 1;
    skip(i);
    if (i < n && p[i] == ']') return 0;  // empty array: parsed.Length == 0 -> false
    bool overflow = false;
    for (;;) {
        skip(i);
        const int64_t len = json_number(p + i, n - i);
        if (len == 0) return 0;
        const float v = to_float(p + i, len);
        if (!std::isfinite(v)) overflow = true;
        out.push_back(v);
        i += len;
        skip(i);
        if (i < n && p[i] == ',') { ++i; continue; }
        if (i < n && p[i] == ']') { ++i; break; }
        return 0;
    }
    skip(i);
    if (i != n) return 0;  // trailing characters after the array: JsonException
    return overflow ? -1 : 1;
}

bool ieq(const unsigned char* p, int64_t n, const char* lit) {
    const int64_t m = (int64_t)strlen(lit);
    if (n != m) return false;
    for (int64_t i = 0; i < n; ++i) {
        unsigned char c = p[i];
        if (c >= 'A' && c <= 'Z') c = (unsigned char)(c + 32);
        if (c != (unsigned char)lit[i]) return false;
    }
    return true;
}

// float.TryParse(s, NumberStyles.Float, InvariantCulture): optional white, sign, digits with an optional '.',
// optional exponent; or NaN / Infinity (any case, .NET Core 3.0+).  Out-of-range magnitudes give +-Infinity.
bool parse_net_float(const unsigned char* p, int64_t n, float* out) {
    while (n > 0 && ws(p[0])) { ++p; --n; }
    while (n > 0 && ws(p[n - 1])) --n;
    if (n == 0) return false;
    {
        const unsigned char* q = p;
        int64_t m = n;
        bool neg = false;
        if (q[0] == '+' || q[0] == '-') { neg = q[0] == '-'; ++q; --m; }
        if (ieq(q, m, "nan")) { *out = NAN; return true; }
        if (ieq(q, m, "infinity")) { *out = neg ? -INFINITY : INFINITY; return true; }
    }
    int64_t i = 0;
    if (p[i] == '+' || p[i] == '-') ++i;
    int64_t nd = 0;
    while (i < n && digit(p[i])) { ++i; ++nd; }
    if (i < n && p[i] == '.') {
        ++i;
        while (i < n && digit(p[i])) { ++i; ++nd; }
    }
    if (nd == 0) return false;
    if (i < n && (p[i] == 'e' || p[i] == 'E')) {
        ++i;
        if (i < n && (p[i] == '+' || p[i] == '-')) ++i;
        if (i >= n || !digit(p[i])) return false;
        while (i < n && digit(p[i])) ++i;
    }
    if (i != n) return false;
    *out = to_float(p, n);
    return true;
}

// TryParseCsvVector (VectorParsing.cs:63-91): Split(',', ' ') with RemoveEmptyEntries | TrimEntries
bool parse_csv(const unsigned char* p, int64_t n, std::vector<float>& out) {
    if (all_white(p, n)) return false;
    int64_t i = 0;
    while (i <= n) {
        int64_t j = i;
        while (j < n && p[j] != ',' && p[j] != ' ') ++j;
        const unsigned char* t = p + i;
        int64_t len = j - i;
        while (len > 0 && ws(t[0])) { ++t; --len; }
        while (len > 0 && ws(t[len - 1])) --len;
        if (len > 0) {
            float v;
            if (!parse_net_float(t, len, &v)) return false;
            out.push_back(v);
        }
        i = j + 1;
    }
    return !out.empty();
}

}  // namespace

extern "C" {

int pyrope_parse_vector(const uint8_t* data, int64_t len, float* out, int64_t cap, int64_t* n_out) {
    if (n_out) *n_out = 0;
    if (!data || len <= 0) return fail(PYROPE_ERR_INVALID_ARG, "Vector payload is empty. (Parameter 'data')");
    std::vector<float> v;
    const int js = parse_json(data, len, v);
    if (js < 0) return fail(PYROPE_ERR_INVALID_ARG, "Either the JSON value is not in a supported format, or is out of bounds for a Single.");
    if (js == 0) {
        v.clear();
        if (!parse_csv(data, len, v)) {
            v.clear();
            if (len % 4 != 0) return fail(PYROPE_ERR_INVALID_ARG, "Unsupported vector format.");
            v.resize((size_t)(len / 4));  // ParseBinaryVector :93-99: the bytes ARE the floats
            memcpy(v.data(), data, (size_t)len);
        }
    }
    if (n_out) *n_out = (int64_t)v.size();
    if (out && cap > 0) memcpy(out, v.data(), sizeof(float) * (size_t)std::min<int64_t>(cap, (int64_t)v.size()));
    return PYROPE_OK;
}

int pyrope_encode_vector(const float* vec, int64_t n, uint8_t* out, int64_t cap_bytes) {
    if (!vec && n > 0) return fail(PYROPE_ERR_INVALID_ARG, "Value cannot be null. (Parameter 'vector')");
    if (n < 0 || cap_bytes < n * 4) return fail(PYROPE_ERR_INVALID_ARG, "destination holds %lld bytes, %lld needed", (long long)cap_bytes, (long long)n * 4);
    if (n > 0) memcpy(out, vec, (size_t)n * 4);  // VectorEncoding.ToLittleEndianBytes: x86-64 / aarch64 are little-endian
    return PYROPE_OK;
}

// FvecsReader.Read: records of int32 d followed by d float32.  limit < 0 = no limit (null); 0 = nothing.
// out may be NULL (count / dimension query).  All records must share one dimension to form a matrix.
int pyrope_fvecs_read(const char* path, int64_t limit, int64_t skip, float* out, int64_t cap_floats, int64_t* count_out,
                      int* dim_out) {
    if (count_out) *count_out = 0;
    if (dim_out) *dim_out = 0;
    if (!path) return fail(PYROPE_ERR_INVALID_ARG, "Value cannot be null. (Parameter 'path')");
    if (limit == 0) return PYROPE_OK;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(PYROPE_ERR_NOT_FOUND, "Could not find file '%s'.", path);
    int64_t count = 0, seen = 0, written = 0;
    int dim0 = 0;
    int rc = PYROPE_OK;
    std::vector<float> rec;
    for (;;) {
        if (limit > 0 && count >= limit) break;
        int32_t d = 0;
        if (fread(&d, 1, 4, f) != 4) break;  // end of file, or a torn header: ReadInt32 throws EndOfStream -> yield break
        if (d <= 0) { rc = fail(PYROPE_ERR_INVALID_ARG, "Invalid vector dimension %d in fvecs file.", d); break; }
        if (dim0 == 0) dim0 = d;
        if (d != dim0) { rc = fail(PYROPE_ERR_DIMENSION, "Vector dimension mismatch"); break; }
        rec.resize((size_t)d);
        if (fread(rec.data(), 4, (size_t)d, f) != (size_t)d) { rc = fail(PYROPE_ERR_INVALID_ARG, "Truncated fvecs record."); break; }
        if (seen++ < skip) continue;
        if (out && written + d <= cap_floats) {
            memcpy(out + written, rec.data(), sizeof(float) * (size_t)d);
            written += d;
        }
        ++count;
    }
    fclose(f);
    if (rc != PYROPE_OK) return rc;
    if (count_out) *count_out = count;
    if (dim_out) *dim_out = dim0;
    return PYROPE_OK;
}

// Stream an fvecs file into an index: 64 MiB batches through pyrope_index_add_batch (labels = row ordinals).
int pyrope_index_add_fvecs(pyrope_index* h, const char* path, int64_t limit, int64_t* added_out) {
    if (added_out) *added_out = 0;
    if (!h) return fail(PYROPE_ERR_INVALID_ARG, "index handle is null");
    if (!path) return fail(PYROPE_ERR_INVALID_ARG, "Value cannot be null. (Parameter 'path')");
    if (limit == 0) return PYROPE_OK;
    int dim = 0;
    TRY(pyrope_index_stats(h, nullptr, nullptr, &dim, nullptr));
    FILE* f = fopen(path, "rb");
    if (!f) return fail(PYROPE_ERR_NOT_FOUND, "Could not find file '%s'.", path);
    const int64_t batch_rows = std::max<int64_t>(1, ((int64_t)64 << 20) / ((int64_t)dim * 4));
    std::vector<float> buf((size_t)batch_rows * dim);
    int64_t added = 0, in_batch = 0;
    auto flush = [&]() -> int {
        if (in_batch == 0) return PYROPE_OK;
        const int r = pyrope_index_add_batch(h, in_batch, buf.data(), nullptr, nullptr);
        if (r == PYROPE_OK) added += in_batch;
        in_batch = 0;
        return r;
    };
    int rc = PYROPE_OK;
    for (;;) {
        if (limit > 0 && added + in_batch >= limit) break;
        int32_t d = 0;
        if (fread(&d, 1, 4, f) != 4) break;
        if (d <= 0) { rc = fail(PYROPE_ERR_INVALID_ARG, "Invalid vector dimension %d in fvecs file.", d); break; }
        if (d != dim) { rc = fail(PYROPE_ERR_DIMENSION, "Vector dimension mismatch"); break; }
        if (fread(buf.data() + (size_t)in_batch * dim, 4, (size_t)d, f) != (size_t)d) { rc = fail(PYROPE_ERR_INVALID_ARG, "Truncated fvecs record."); break; }
        if (++in_batch == batch_rows && (rc = flush()) != PYROPE_OK) break;
    }
    fclose(f);
    if (rc == PYROPE_OK) rc = flush();
    if (added_out) *added_out = added;
    return rc;
}

}  // extern "C"
