// pa_mzml_index: the XML structure of an mzML file -> retained spectra and the byte ranges of their binary arrays.
//
// Same records as the stdlib reader (pyascore_b200/parsing/_xml.py iter_mzml + SpectraParser._records/_get_spectra,
// reference: spec_parsers.py:49-110, :175-282), without touching a payload: base64 text holds no '<', so one memchr
// per tag walks the file.  What the stdlib path would read differently from the raw bytes (markup or entities inside
// <binary>, a DOCTYPE internal subset) or what the device layout needs (array lengths) is refused with a reason.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/pyascore_b200.h"

namespace {

struct Refuse {
    std::string text;
};

[[noreturn]] void refuse(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    throw Refuse{buf};
}

struct Param {
    std::string acc, value;
    bool has_value;
};

struct ArrayRec {
    std::vector<Param> params;
    std::vector<std::string> refs;
    std::string array_length;
    bool has_array_length = false;
    bool has_binary = false;
    bool markup = false;              // comment, CDATA or an element inside <binary>
    int64_t text_off = 0, text_len = 0;
};

struct Spectrum {
    std::string id, default_len;
    bool has_default_len = false;
    std::vector<Param> params;
    std::vector<std::string> refs;
    int pl_state = 0;                 // 0 no precursorList yet, 1 inside the first one, 2 done
    std::string pl_count;
    bool has_pl_count = false;
    int n_prec = 0;
    bool sil_seen = false, ion_seen = false, ion_open = false, sil_open = false, prec_open = false;
    std::unordered_map<std::string, Param> ion;    // cvParams of the first selectedIon (last accession wins)
    int bl_state = 0;                 // 0 no binaryDataArrayList yet, 1 inside the first one, 2 done
    std::vector<ArrayRec> arrays;
    bool bda_open = false, binary_seen = false;
};

struct Record {
    int64_t scan;
    int32_t ms_level;
    double pmz;
    int32_t pz;
    int64_t count;                    // peaks (0 without both arrays)
    ArrayRec mz, inten;
    int mz_dtype, in_dtype;
    bool mz_zlib, in_zlib;
    bool has_arrays;                  // both arrays present: two table entries, even for zero peaks
};

struct Index {
    pa_mzml_index_t pub;
    std::vector<int64_t> scan, spec_off;
    std::vector<int32_t> ms_level, pz;
    std::vector<double> pmz;
    std::vector<pa_mzml_array> arrays;
};

inline bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r'; }

std::string strip(const std::string& s) {
    size_t a = 0, b = s.size();
    while (a < b && (is_ws(s[a]) || s[a] == '\f' || s[a] == '\v')) a++;
    while (b > a && (is_ws(s[b - 1]) || s[b - 1] == '\f' || s[b - 1] == '\v')) b--;
    return s.substr(a, b - a);
}

// Python int(text) for plain decimal text (surrounding whitespace, one sign); anything else refused
bool py_int(const std::string& text, int64_t& out) {
    const std::string s = strip(text);
    size_t i = 0;
    bool neg = false;
    if (i < s.size() && (s[i] == '+' || s[i] == '-')) neg = s[i++] == '-';
    if (i == s.size()) return false;
    unsigned long long v = 0;
    for (; i < s.size(); i++) {
        if (s[i] < '0' || s[i] > '9') return false;
        if (v > (9223372036854775807ull - (unsigned)(s[i] - '0')) / 10) return false;
        v = v * 10 + (unsigned)(s[i] - '0');
    }
    out = neg ? -(int64_t)v : (int64_t)v;
    return true;
}

// Python float(text): decimal, inf/infinity/nan; strtod is correctly rounded like Python's parser.  Hex and
// underscore forms (which the two parse differently) are refused.
bool py_float(const std::string& text, double& out) {
    const std::string s = strip(text);
    if (s.empty() || s.find_first_of("xX_()") != std::string::npos) return false;
    char* end = nullptr;
    out = strtod(s.c_str(), &end);
    return end == s.c_str() + s.size();
}

void append_utf8(std::string& o, unsigned long cp) {
    if (cp < 0x80) o += (char)cp;
    else if (cp < 0x800) { o += (char)(0xC0 | (cp >> 6)); o += (char)(0x80 | (cp & 63)); }
    else if (cp < 0x10000) { o += (char)(0xE0 | (cp >> 12)); o += (char)(0x80 | ((cp >> 6) & 63)); o += (char)(0x80 | (cp & 63)); }
    else { o += (char)(0xF0 | (cp >> 18)); o += (char)(0x80 | ((cp >> 12) & 63)); o += (char)(0x80 | ((cp >> 6) & 63)); o += (char)(0x80 | (cp & 63)); }
}

// attribute value as the XML parser reports it: entities decoded, literal tab / newline / CR normalised to spaces
std::string attr_value(const char* a, const char* b) {
    std::string o;
    o.reserve((size_t)(b - a));
    for (const char* p = a; p < b; p++) {
        if (*p == '&') {
            const char* semi = (const char*)memchr(p, ';', (size_t)(b - p));
            if (!semi) refuse("malformed entity in an attribute value");
            const std::string ent(p + 1, semi);
            if (ent == "lt") o += '<';
            else if (ent == "gt") o += '>';
            else if (ent == "amp") o += '&';
            else if (ent == "quot") o += '"';
            else if (ent == "apos") o += '\'';
            else if (ent.size() > 1 && ent[0] == '#') {
                char* e = nullptr;
                const unsigned long cp = (ent[1] == 'x') ? strtoul(ent.c_str() + 2, &e, 16) : strtoul(ent.c_str() + 1, &e, 10);
                if (*e || ent.size() == (ent[1] == 'x' ? 2u : 1u) || cp == 0 || cp > 0x10FFFF) refuse("bad character reference &%s;", ent.c_str());
                append_utf8(o, cp);
            } else refuse("undefined entity &%s; in an attribute value", ent.c_str());
            p = semi;
        } else if (*p == '\t' || *p == '\n' || *p == '\r') {
            o += ' ';
        } else o += *p;
    }
    return o;
}

struct Tag {
    const char* name;
    size_t name_len;
    std::vector<std::pair<std::string, std::string>> attrs;
    bool self_closing;
    const char* end;                  // one past '>'
};

std::string local(const char* name, size_t n) {
    const void* colon = memchr(name, ':', n);
    if (!colon) return std::string(name, n);
    const char* c = (const char*)colon + 1;
    return std::string(c, name + n);
}

bool find_attr(const Tag& t, const char* name, std::string& out) {
    for (auto& kv : t.attrs)
        if (kv.first == name) { out = kv.second; return true; }
    return false;
}

const char* find_seq(const char* p, const char* end, const char* seq) {
    const size_t n = strlen(seq);
    while (p < end) {
        const char* q = (const char*)memchr(p, seq[0], (size_t)(end - p));
        if (!q || (size_t)(end - q) < n) return nullptr;
        if (memcmp(q, seq, n) == 0) return q;
        p = q + 1;
    }
    return nullptr;
}

// start tag at p ('<' + name): name, attributes (both quote styles), '/>' or '>'
Tag parse_start(const char* p, const char* end) {
    Tag t;
    const char* q = p + 1;
    while (q < end && !is_ws(*q) && *q != '>' && *q != '/') q++;
    t.name = p + 1;
    t.name_len = (size_t)(q - (p + 1));
    if (t.name_len == 0) refuse("malformed tag at byte %lld", (long long)0);
    for (;;) {
        while (q < end && is_ws(*q)) q++;
        if (q >= end) refuse("unterminated tag");
        if (*q == '>') { t.self_closing = false; t.end = q + 1; return t; }
        if (*q == '/') {
            if (q + 1 < end && q[1] == '>') { t.self_closing = true; t.end = q + 2; return t; }
            refuse("malformed tag");
        }
        const char* n0 = q;
        while (q < end && !is_ws(*q) && *q != '=' && *q != '>' && *q != '/') q++;
        const std::string name = local(n0, (size_t)(q - n0));
        while (q < end && is_ws(*q)) q++;
        if (q >= end || *q != '=') refuse("attribute without a value");
        q++;
        while (q < end && is_ws(*q)) q++;
        if (q >= end || (*q != '"' && *q != '\'')) refuse("unquoted attribute value");
        const char quote = *q++;
        const char* v1 = (const char*)memchr(q, quote, (size_t)(end - q));
        if (!v1) refuse("unterminated attribute value");
        t.attrs.emplace_back(name, attr_value(q, v1));
        q = v1 + 1;
    }
}

enum Dtype { DT_NONE = -1 };

int dtype_of(const std::string& acc) {
    if (acc == "MS:1000523") return PA_MZML_F64;
    if (acc == "MS:1000521") return PA_MZML_F32;
    if (acc == "MS:1000519") return PA_MZML_I32;
    if (acc == "MS:1000522") return PA_MZML_I64;
    return DT_NONE;
}

bool is_numpress(const std::string& acc) {
    return acc == "MS:1002312" || acc == "MS:1002313" || acc == "MS:1002314" || acc == "MS:1002746" || acc == "MS:1002747" ||
           acc == "MS:1002748";
}

class Indexer {
public:
    Indexer(const char* buf, int64_t n, int32_t ms_level) : buf_(buf), end_(buf + n), want_level_(ms_level) {}

    void run() {
        const char* p = buf_;
        if (end_ - p >= 2 && ((uint8_t)p[0] == 0xFF || (uint8_t)p[0] == 0xFE || p[0] == 0 || p[1] == 0))
            refuse("not a UTF-8 file");
        while (p < end_) {
            const char* lt = (const char*)memchr(p, '<', (size_t)(end_ - p));
            if (!lt) break;
            if (in_binary_ && !starts(lt, "</")) binary_markup();
            if (starts(lt, "<!--")) {
                const char* e = find_seq(lt + 4, end_, "-->");
                if (!e) refuse("unterminated comment");
                p = e + 3;
            } else if (starts(lt, "<![CDATA[")) {
                const char* e = find_seq(lt + 9, end_, "]]>");
                if (!e) refuse("unterminated CDATA section");
                p = e + 3;
            } else if (starts(lt, "<?")) {
                const char* e = find_seq(lt + 2, end_, "?>");
                if (!e) refuse("unterminated processing instruction");
                p = e + 2;
            } else if (starts(lt, "<!")) {
                const char* e = (const char*)memchr(lt, '>', (size_t)(end_ - lt));
                if (!e) refuse("unterminated declaration");
                if (memchr(lt, '[', (size_t)(e - lt))) refuse("a DOCTYPE internal subset (entity declarations) is not read by this path");
                p = e + 1;
            } else if (lt + 1 < end_ && lt[1] == '/') {
                const char* e = (const char*)memchr(lt, '>', (size_t)(end_ - lt));
                if (!e) refuse("unterminated end tag");
                const char* n1 = e;
                while (n1 > lt + 2 && is_ws(n1[-1])) n1--;
                end_element(lt, lt + 2, (size_t)(n1 - (lt + 2)));
                p = e + 1;
            } else {
                Tag t = parse_start(lt, end_);
                start_element(t);
                if (t.self_closing) end_element(nullptr, t.name, t.name_len);
                p = t.end;
            }
        }
        if (!stack_.empty()) refuse("the file ends inside <%s>", stack_.back().c_str());
    }

    std::vector<Record> records;

private:
    const char* buf_;
    const char* end_;
    int32_t want_level_;
    std::vector<std::string> stack_;     // raw (prefixed) names of the open elements
    std::vector<std::string> locals_;
    std::unordered_map<std::string, std::vector<Param>> groups_;
    int grp_depth_ = -1;
    std::string grp_id_;
    std::vector<Param> grp_params_;
    int sp_depth_ = -1;
    Spectrum sp_;
    bool in_binary_ = false;

    bool starts(const char* p, const char* s) const {
        const size_t n = strlen(s);
        return (size_t)(end_ - p) >= n && memcmp(p, s, n) == 0;
    }

    void binary_markup() {
        sp_.arrays.back().markup = true;
        in_binary_ = false;
    }

    static Param param_of(const Tag& t) {
        Param pr;
        find_attr(t, "accession", pr.acc);
        pr.has_value = find_attr(t, "value", pr.value);
        return pr;
    }

    void start_element(const Tag& t) {
        const std::string name = local(t.name, t.name_len);
        const int depth = (int)stack_.size();        // depth of this element
        if (grp_depth_ >= 0 && depth == grp_depth_ + 1 && name == "cvParam") grp_params_.push_back(param_of(t));
        if (name == "referenceableParamGroup" && grp_depth_ < 0) {
            grp_depth_ = depth;
            grp_id_.clear();
            find_attr(t, "id", grp_id_);
            grp_params_.clear();
        }
        if (sp_depth_ >= 0) spectrum_child(t, name, depth);
        if (name == "spectrum" && sp_depth_ < 0) {
            sp_depth_ = depth;
            sp_ = Spectrum();
            find_attr(t, "id", sp_.id);
            sp_.has_default_len = find_attr(t, "defaultArrayLength", sp_.default_len);
        }
        stack_.emplace_back(t.name, t.name_len);
        locals_.push_back(name);
    }

    void spectrum_child(const Tag& t, const std::string& name, int depth) {
        const int rel = depth - sp_depth_;
        if (rel == 1) {
            if (name == "cvParam") sp_.params.push_back(param_of(t));
            else if (name == "referenceableParamGroupRef") { std::string r; find_attr(t, "ref", r); sp_.refs.push_back(r); }
            else if (name == "precursorList" && sp_.pl_state == 0) {
                sp_.pl_state = 1;
                sp_.has_pl_count = find_attr(t, "count", sp_.pl_count);
            } else if (name == "binaryDataArrayList" && sp_.bl_state == 0) sp_.bl_state = 1;
            return;
        }
        const std::string& parent = locals_.back();
        if (sp_.pl_state == 1) {
            if (rel == 2 && name == "precursor") { if (++sp_.n_prec == 1) sp_.prec_open = true; }
            else if (rel == 3 && sp_.prec_open && name == "selectedIonList" && !sp_.sil_seen && parent == "precursor") {
                sp_.sil_seen = sp_.sil_open = true;
            } else if (rel == 4 && sp_.sil_open && name == "selectedIon" && !sp_.ion_seen && parent == "selectedIonList") {
                sp_.ion_seen = sp_.ion_open = true;
            } else if (rel == 5 && sp_.ion_open && name == "cvParam" && parent == "selectedIon") {
                Param pr = param_of(t);
                sp_.ion[pr.acc] = pr;
            }
        }
        if (sp_.bl_state == 1) {
            if (rel == 2 && name == "binaryDataArray") {
                sp_.arrays.emplace_back();
                sp_.bda_open = true;
                sp_.binary_seen = false;
                sp_.arrays.back().has_array_length = find_attr(t, "arrayLength", sp_.arrays.back().array_length);
            } else if (rel == 3 && sp_.bda_open && parent == "binaryDataArray") {
                ArrayRec& a = sp_.arrays.back();
                if (name == "cvParam") a.params.push_back(param_of(t));
                else if (name == "referenceableParamGroupRef") { std::string r; find_attr(t, "ref", r); a.refs.push_back(r); }
                else if (name == "binary" && !sp_.binary_seen) {
                    sp_.binary_seen = true;
                    a.has_binary = true;
                    a.text_off = t.end - buf_;
                    in_binary_ = !t.self_closing;
                }
            }
        }
    }

    void end_element(const char* tag_start, const char* name, size_t n) {
        if (stack_.empty() || stack_.back().size() != n || memcmp(stack_.back().data(), name, n) != 0)
            refuse("mismatched end tag </%.*s>", (int)n, name);
        const int depth = (int)stack_.size() - 1;
        const std::string lname = locals_.back();
        stack_.pop_back();
        locals_.pop_back();
        if (in_binary_ && lname == "binary") {
            sp_.arrays.back().text_len = (tag_start - buf_) - sp_.arrays.back().text_off;
            in_binary_ = false;
        }
        if (depth == grp_depth_) {
            groups_[grp_id_] = grp_params_;
            grp_depth_ = -1;
        }
        if (sp_depth_ >= 0 && depth > sp_depth_) {
            const int rel = depth - sp_depth_;
            if (rel == 1 && lname == "precursorList" && sp_.pl_state == 1) sp_.pl_state = 2;
            else if (rel == 1 && lname == "binaryDataArrayList" && sp_.bl_state == 1) sp_.bl_state = 2;
            else if (rel == 2 && lname == "precursor") sp_.prec_open = false;
            else if (rel == 3 && lname == "selectedIonList") sp_.sil_open = false;
            else if (rel == 4 && lname == "selectedIon") sp_.ion_open = false;
            else if (rel == 2 && lname == "binaryDataArray") sp_.bda_open = false;
        }
        if (depth == sp_depth_) {
            finish_spectrum();
            sp_depth_ = -1;
        }
    }

    std::vector<Param> resolved(const std::vector<Param>& direct, const std::vector<std::string>& refs) const {
        std::vector<Param> out = direct;
        for (auto& r : refs) {
            auto it = groups_.find(r);
            if (it != groups_.end()) out.insert(out.end(), it->second.begin(), it->second.end());
        }
        return out;
    }

    void finish_spectrum() {
        Record rec{};
        // scan: first "scan=" followed by a digit, as re.search((?<=scan=)[0-9]+) finds it
        rec.scan = -1;
        for (size_t at = sp_.id.find("scan="); at != std::string::npos; at = sp_.id.find("scan=", at + 1)) {
            size_t d = at + 5, e = d;
            while (e < sp_.id.size() && sp_.id[e] >= '0' && sp_.id[e] <= '9') e++;
            if (e > d) {
                int64_t v;
                if (!py_int(sp_.id.substr(d, e - d), v)) refuse("scan number %s does not fit 64 bits", sp_.id.substr(d, e - d).c_str());
                rec.scan = v;
                break;
            }
        }
        int64_t level = 0;
        for (auto& pr : resolved(sp_.params, sp_.refs))
            if (pr.acc == "MS:1000511") {
                if (!pr.has_value || !py_int(pr.value, level) || level != (int32_t)level)
                    refuse("ms level %s of spectrum '%s' is not an integer", pr.value.c_str(), sp_.id.c_str());
            }
        rec.ms_level = (int32_t)level;
        rec.pmz = NAN;
        rec.pz = 0;
        if (sp_.pl_state != 0) {
            int64_t count = sp_.n_prec;
            if (sp_.has_pl_count && !py_int(sp_.pl_count, count)) refuse("precursorList count %s is not an integer", sp_.pl_count.c_str());
            if (count > 1) refuse("Multiple precursors not supported at this time");
            if (sp_.ion_seen) {
                // both keys must exist; a missing value attribute reads as missing (TypeError in the stdlib reader)
                auto a = sp_.ion.find("MS:1000744"), b = sp_.ion.find("MS:1000041");
                if (a != sp_.ion.end() && a->second.has_value) {
                    double mz;
                    if (!py_float(a->second.value, mz)) refuse("precursor m/z %s is not a number", a->second.value.c_str());
                    if (b != sp_.ion.end() && b->second.has_value) {
                        int64_t z;
                        if (!py_int(b->second.value, z) || z != (int32_t)z) refuse("precursor charge %s is not a 32-bit integer", b->second.value.c_str());
                        rec.pmz = mz;
                        rec.pz = (int32_t)z;
                    }
                }
            }
        }
        // arrays: numpress raises for every array (also of dropped levels); the last m/z and intensity arrays win
        const ArrayRec* mz = nullptr;
        const ArrayRec* in = nullptr;
        int mz_dt = DT_NONE, in_dt = DT_NONE;
        bool mz_zl = false, in_zl = false;
        for (auto& a : sp_.arrays) {
            int dt = DT_NONE, kind = 0;
            bool zl = false;
            for (auto& pr : resolved(a.params, a.refs)) {
                const int d = dtype_of(pr.acc);
                if (d != DT_NONE) dt = d;
                else if (pr.acc == "MS:1000574") zl = true;
                else if (is_numpress(pr.acc))
                    refuse("mzML numpress compression (%s) is not supported by the stdlib reader", pr.acc.c_str());
                else if (pr.acc == "MS:1000514") kind = 1;
                else if (pr.acc == "MS:1000515") kind = 2;
            }
            if (kind == 0 || dt == DT_NONE) continue;
            if (kind == 1) { mz = &a; mz_dt = dt; mz_zl = zl; }
            else { in = &a; in_dt = dt; in_zl = zl; }
        }
        if (want_level_ && rec.ms_level != want_level_) return;
        rec.count = 0;
        if (mz && in) {
            int64_t cm, ci;
            if (!count_of(*mz, cm) || !count_of(*in, ci))
                refuse("spectrum '%s': a binary array without a usable arrayLength / defaultArrayLength", sp_.id.c_str());
            if (cm != ci) refuse("spectrum '%s': %lld m/z values but %lld intensities", sp_.id.c_str(), (long long)cm, (long long)ci);
            if (mz->markup || in->markup) refuse("spectrum '%s': markup (comment, CDATA, element) inside <binary>", sp_.id.c_str());
            rec.count = cm;
            rec.has_arrays = true;
            rec.mz = *mz;
            rec.inten = *in;
            rec.mz_dtype = mz_dt;
            rec.in_dtype = in_dt;
            rec.mz_zlib = mz_zl;
            rec.in_zlib = in_zl;
        }
        records.push_back(std::move(rec));
    }

    bool count_of(const ArrayRec& a, int64_t& c) const {
        const bool ok = a.has_array_length ? py_int(a.array_length, c) : (sp_.has_default_len && py_int(sp_.default_len, c));
        return ok && c >= 0;
    }
};

}  // namespace

// spec_parsers.py:49-110 (MzMLExtractor's XML half) and :175-282 (SpectraParser's level filter and scan sort)
extern "C" int pa_mzml_index(const uint8_t* bytes, int64_t n, int32_t ms_level, pa_mzml_index_t** out, char* err,
                             int32_t err_cap) {
    if (err && err_cap > 0) err[0] = 0;
    if (!out || (!bytes && n > 0) || n < 0) {
        if (err && err_cap > 0) snprintf(err, (size_t)err_cap, "pa_mzml_index: NULL or negative argument");
        return PA_ERR_ARG;
    }
    *out = nullptr;
    try {
        Indexer ix((const char*)bytes, n, ms_level);
        ix.run();
        std::vector<Record>& recs = ix.records;
        std::stable_sort(recs.begin(), recs.end(), [](const Record& a, const Record& b) { return a.scan < b.scan; });
        Index* idx = new Index();
        const size_t ns = recs.size();
        idx->scan.resize(ns);
        idx->ms_level.resize(ns);
        idx->pmz.resize(ns);
        idx->pz.resize(ns);
        idx->spec_off.assign(ns + 1, 0);
        for (size_t i = 0; i < ns; i++) {
            const Record& r = recs[i];
            idx->scan[i] = r.scan;
            idx->ms_level[i] = r.ms_level;
            idx->pmz[i] = r.pmz;
            idx->pz[i] = r.pz;
            idx->spec_off[i + 1] = idx->spec_off[i] + r.count;
            if (!r.has_arrays) continue;
            pa_mzml_array m{r.mz.text_off, r.mz.text_len, idx->spec_off[i], r.count, (int64_t)i, r.mz_dtype, r.mz_zlib ? PA_MZML_ZLIB : 0};
            pa_mzml_array t{r.inten.text_off, r.inten.text_len, idx->spec_off[i], r.count, (int64_t)i, r.in_dtype,
                            (r.in_zlib ? PA_MZML_ZLIB : 0) | PA_MZML_INTENSITY};
            idx->arrays.push_back(m);
            idx->arrays.push_back(t);
        }
        idx->pub = pa_mzml_index_t{(int64_t)ns, idx->scan.data(), idx->ms_level.data(), idx->pmz.data(), idx->pz.data(),
                                   idx->spec_off.data(), (int64_t)idx->arrays.size(), idx->arrays.data()};
        *out = &idx->pub;
        return PA_OK;
    } catch (const Refuse& r) {
        if (err && err_cap > 0) snprintf(err, (size_t)err_cap, "%s", r.text.c_str());
        return PA_ERR_ARG;
    } catch (const std::bad_alloc&) {
        if (err && err_cap > 0) snprintf(err, (size_t)err_cap, "pa_mzml_index: out of host memory");
        return PA_ERR_ARG;
    }
}

extern "C" void pa_mzml_index_free(pa_mzml_index_t* index) {
    // pub is the first member of Index
    delete reinterpret_cast<Index*>(index);
}
