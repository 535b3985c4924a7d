// wavfile.cpp — WAV / RF64 containers either side of the chain (SURVEY.md 8(f) rank 4).
//
// The reference reads WAV captures through libsndfile (src/input_wav.c:542-632: sf_open, 2 channels,
// PCM_16 -> cs16 / PCM_U8 -> cu8, rate from the header, sf_read_raw of 16384-frame chunks :667), pulls SDR
// metadata out of the first `auxi` chunk (XML attributes of <Definition> through expat :345-441, else the
// SDRuno binary layout :294-332) and out of the file name (:190-271), and can turn the recorded centre
// frequency into the chain's NCO shift (--wav-center-target-freq :612-629).  It writes WAV / RF64 with
// sf_write_raw and lets libsndfile patch the sizes on close (src/output_wav_common.c:54-174).
//
// Neither libsndfile nor expat is used here: the RIFF / RF64 chunk walk, the handful of XML the auxi chunk
// needs and the two headers are written out in plain C++.  The payload goes through iqio::run_stream
// (rawfile.cpp) — large pinned reads, one chain call per chunk train, one write per train.  Everything in this
// file except iqgpu_wavfile_run is host-only and works without a device.
#include <cctype>
#include <cerrno>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <string>
#include <utility>
#include <vector>

#include "../../include/iqgpu.h"
#include "stream_io.hpp"

namespace {

constexpr size_t kMaxMetadataChunk = 1024 * 1024;   // MAX_METADATA_CHUNK_SIZE, src/input_wav.c:42

uint16_t le16(const unsigned char* p) { return (uint16_t)(p[0] | (p[1] << 8)); }
uint32_t le32(const unsigned char* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
uint64_t le64(const unsigned char* p) { return (uint64_t)le32(p) | ((uint64_t)le32(p + 4) << 32); }
void put16(unsigned char* p, uint32_t v) { p[0] = (unsigned char)v; p[1] = (unsigned char)(v >> 8); }
void put32(unsigned char* p, uint32_t v) { put16(p, v); put16(p + 2, v >> 16); }
void put64(unsigned char* p, uint64_t v) { put32(p, (uint32_t)v); put32(p + 4, (uint32_t)(v >> 32)); }

// snprintf(dst, cap, "%s", src) of the reference's string attributes: truncating, always terminated
void copy_text(char* dst, size_t cap, const std::string& src)
{
    const size_t n = src.size() < cap - 1 ? src.size() : cap - 1;
    memcpy(dst, src.data(), n);
    dst[n] = '\0';
}

// UTC calendar time -> seconds; the reference's timegm_portable (src/input_wav.c:273-292) is mktime under TZ="",
// i.e. timegm with its field normalisation
bool utc_seconds(int year, int month, int day, int hour, int min, int sec, int64_t* out)
{
    struct tm t;
    memset(&t, 0, sizeof(t));
    t.tm_year = year - 1900; t.tm_mon = month - 1; t.tm_mday = day;
    t.tm_hour = hour; t.tm_min = min; t.tm_sec = sec;
    const time_t ts = timegm(&t);
    if (ts == (time_t)-1) return false;
    *out = (int64_t)ts;
    return true;
}

// ---- the XML the auxi chunk needs: start tags with their attributes, in document order -------------------------------
// expat semantics that matter to the reference: handlers fire for every start tag before the first
// well-formedness error, and the return value of XML_Parse is ignored (src/input_wav.c:418).
struct XmlStartTag {
    std::string name;
    std::vector<std::pair<std::string, std::string>> attrs;
};

// A cursor over the chunk that yields XML characters (UTF-8, or ISO-8859-1 when the declaration says so)
struct XmlSource {
    const unsigned char* d;
    size_t n;
    bool latin1 = false;

    // code point at i and its byte length; 0 = end of data, malformed UTF-8, or a character XML does not allow
    int at(size_t i, uint32_t* cp) const
    {
        if (i >= n) return 0;
        const unsigned char c = d[i];
        uint32_t v;
        int len;
        if (c < 0x80 || latin1) { v = c; len = 1; }
        else if (c >= 0xC2 && c <= 0xDF) { v = c & 0x1F; len = 2; }
        else if (c >= 0xE0 && c <= 0xEF) { v = c & 0x0F; len = 3; }
        else if (c >= 0xF0 && c <= 0xF4) { v = c & 0x07; len = 4; }
        else return 0;
        if (i + len > n) return 0;
        for (int k = 1; k < len; k++) {
            if ((d[i + k] & 0xC0) != 0x80) return 0;
            v = (v << 6) | (d[i + k] & 0x3F);
        }
        if ((len == 3 && v < 0x800) || (len == 4 && (v < 0x10000 || v > 0x10FFFF))) return 0;
        const bool allowed = v == 0x9 || v == 0xA || v == 0xD || (v >= 0x20 && v <= 0xD7FF) || (v >= 0xE000 && v <= 0xFFFD) || v >= 0x10000;
        if (!allowed) return 0;
        *cp = v;
        return len;
    }
};

bool is_xml_space(uint32_t c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r'; }
// Name characters: exact for ASCII and Latin-1, by block beyond (letters and ideographs in, punctuation / symbols /
// private use / specials out) — metadata writers use ASCII names
bool is_name_start(uint32_t c)
{
    if (c < 0x80) return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z') || c == '_' || c == ':';
    if (c < 0x100) return c >= 0xC0 && c != 0xD7 && c != 0xF7;
    if (c >= 0x2000 && c <= 0x2FFF) return c == 0x2126 || (c >= 0x212A && c <= 0x212B) || c == 0x212E || (c >= 0x2180 && c <= 0x2182);
    if (c >= 0x3000 && c <= 0x3006) return false;
    if (c >= 0xD7A4 && c <= 0xFFFF) return false;
    return c < 0x10000;
}
bool is_name_char(uint32_t c) { return is_name_start(c) || (c >= '0' && c <= '9') || c == '-' || c == '.' || c == 0xB7; }

void append_utf8(std::string& s, uint32_t cp)
{
    if (cp < 0x80) s += (char)cp;
    else if (cp < 0x800) { s += (char)(0xC0 | (cp >> 6)); s += (char)(0x80 | (cp & 0x3F)); }
    else if (cp < 0x10000) { s += (char)(0xE0 | (cp >> 12)); s += (char)(0x80 | ((cp >> 6) & 0x3F)); s += (char)(0x80 | (cp & 0x3F)); }
    else { s += (char)(0xF0 | (cp >> 18)); s += (char)(0x80 | ((cp >> 12) & 0x3F)); s += (char)(0x80 | ((cp >> 6) & 0x3F)); s += (char)(0x80 | (cp & 0x3F)); }
}

// "&name;" / "&#n;" / "&#xh;" at i (src[i] == '&'): appends the replacement text, returns the byte length or 0
size_t reference_at(const XmlSource& src, size_t i, std::string* out)
{
    size_t j = i + 1;
    std::string body;
    while (j < src.n && src.d[j] != ';' && body.size() < 12) body += (char)src.d[j++];
    if (j >= src.n || src.d[j] != ';' || body.empty()) return 0;
    uint32_t cp;
    if (body == "amp") cp = '&';
    else if (body == "lt") cp = '<';
    else if (body == "gt") cp = '>';
    else if (body == "quot") cp = '"';
    else if (body == "apos") cp = '\'';
    else if (body[0] == '#') {
        const bool hex = body.size() > 1 && body[1] == 'x';
        const char* digits = body.c_str() + (hex ? 2 : 1);
        if (!*digits) return 0;
        for (const char* p = digits; *p; p++)
            if (!((*p >= '0' && *p <= '9') || (hex && ((*p >= 'a' && *p <= 'f') || (*p >= 'A' && *p <= 'F'))))) return 0;
        const unsigned long v = strtoul(digits, nullptr, hex ? 16 : 10);
        const bool allowed = v == 0x9 || v == 0xA || v == 0xD || (v >= 0x20 && v <= 0xD7FF) || (v >= 0xE000 && v <= 0xFFFD) || (v >= 0x10000 && v <= 0x10FFFF);
        if (!allowed) return 0;
        cp = (uint32_t)v;
    } else return 0;                                        // no DTD: any other entity is undefined
    if (out) append_utf8(*out, cp);
    return j + 1 - i;
}

// a Name at i: its byte length (0 = none), text appended to *out
size_t name_at(const XmlSource& src, size_t i, std::string* out)
{
    uint32_t cp;
    int len = src.at(i, &cp);
    if (!len || !is_name_start(cp)) return 0;
    size_t j = i;
    while ((len = src.at(j, &cp)) != 0 && is_name_char(cp)) {
        if (out) append_utf8(*out, cp);
        j += len;
    }
    return j - i;
}

// every character up to (not including) the terminator string is an allowed XML character; returns the offset of the
// terminator or npos
size_t find_terminator(const XmlSource& src, size_t i, const char* term)
{
    const size_t tl = strlen(term);
    while (i < src.n) {
        if (i + tl <= src.n && memcmp(src.d + i, term, tl) == 0) return i;
        uint32_t cp;
        const int len = src.at(i, &cp);
        if (!len) return (size_t)-1;
        i += len;
    }
    return (size_t)-1;
}

// <?xml version="1.x" [encoding="..."] [standalone="yes|no"] ?> at the very start; sets latin1; false = malformed / unsupported
bool xml_declaration(XmlSource& src, size_t i, size_t* end)
{
    size_t j = i + 5;
    const char* expected[] = {"version", "encoding", "standalone"};
    int next = 0;
    for (;;) {
        const size_t before = j;
        while (j < src.n && is_xml_space(src.d[j])) j++;
        if (j + 1 < src.n && src.d[j] == '?' && src.d[j + 1] == '>') { *end = j + 2; return next >= 1; }
        if (j == before) return false;
        std::string key, value;
        const size_t kl = name_at(src, j, &key);
        if (!kl) return false;
        j += kl;
        while (j < src.n && is_xml_space(src.d[j])) j++;
        if (j >= src.n || src.d[j] != '=') return false;
        j++;
        while (j < src.n && is_xml_space(src.d[j])) j++;
        if (j >= src.n || (src.d[j] != '"' && src.d[j] != '\'')) return false;
        const unsigned char q = src.d[j++];
        while (j < src.n && src.d[j] != q) value += (char)src.d[j++];
        if (j >= src.n) return false;
        j++;
        while (next < 3 && key != expected[next]) { if (next == 0) return false; next++; }
        if (next >= 3) return false;
        if (next == 0) {
            for (char c : value)           // expat checks the alphabet of the version, not its value
                if (!isalnum((unsigned char)c) && c != '.' && c != '_' && c != ':' && c != '-') return false;
        } else if (next == 1) {
            std::string enc;
            for (char c : value) enc += (char)tolower((unsigned char)c);
            if (enc == "iso-8859-1") src.latin1 = true;
            else if (enc != "utf-8" && enc != "us-ascii") return false;      // UTF-16 and friends: not handled here
        } else if (value != "yes" && value != "no") return false;
        next++;
    }
}

std::vector<XmlStartTag> scan_xml_start_tags(const unsigned char* data, size_t n)
{
    std::vector<XmlStartTag> tags;
    XmlSource src{data, n};
    std::vector<std::string> open;                         // element stack
    bool root_closed = false;
    size_t i = 0;
    if (n >= 3 && data[0] == 0xEF && data[1] == 0xBB && data[2] == 0xBF) i = 3;         // UTF-8 byte order mark
    if (i + 5 < n && memcmp(data + i, "<?xml", 5) == 0 && is_xml_space(data[i + 5])) {
        if (!xml_declaration(src, i, &i)) return tags;
    }
    while (i < n) {
        if (data[i] != '<') {
            uint32_t cp;
            const int len = src.at(i, &cp);
            if (!len) return tags;
            if (open.empty()) { if (!is_xml_space(cp)) return tags; }                  // only white space outside the root
            else if (cp == '&') { const size_t r = reference_at(src, i, nullptr); if (!r) return tags; i += r; continue; }
            else if (cp == ']' && i + 2 < n && data[i + 1] == ']' && data[i + 2] == '>') return tags;
            i += len;
            continue;
        }
        if (i + 1 >= n) return tags;
        if (data[i + 1] == '?') {                                                       // processing instruction
            std::string target;
            const size_t tl = name_at(src, i + 2, &target);
            if (!tl) return tags;
            std::string low;
            for (char c : target) low += (char)tolower((unsigned char)c);
            if (low == "xml") return tags;                                              // the declaration is only legal at the start
            size_t j = i + 2 + tl;
            if (!(j + 1 < n && data[j] == '?' && data[j + 1] == '>') && !(j < n && is_xml_space(data[j]))) return tags;
            const size_t e = find_terminator(src, j, "?>");
            if (e == (size_t)-1) return tags;
            i = e + 2;
            continue;
        }
        if (data[i + 1] == '!') {
            if (i + 3 < n && data[i + 2] == '-' && data[i + 3] == '-') {                // comment: no "--" inside
                const size_t e = find_terminator(src, i + 4, "--");
                if (e == (size_t)-1 || e + 2 >= n || data[e + 2] != '>') return tags;
                i = e + 3;
                continue;
            }
            if (!open.empty() && i + 9 <= n && memcmp(data + i, "<![CDATA[", 9) == 0) {
                const size_t e = find_terminator(src, i + 9, "]]>");
                if (e == (size_t)-1) return tags;
                i = e + 3;
                continue;
            }
            return tags;                                                                // DOCTYPE and the rest: not in metadata chunks
        }
        if (data[i + 1] == '/') {                                                       // end tag: must close the innermost element
            std::string name;
            const size_t nl = name_at(src, i + 2, &name);
            size_t j = i + 2 + nl;
            while (j < n && is_xml_space(data[j])) j++;
            if (!nl || j >= n || data[j] != '>' || open.empty() || open.back() != name) return tags;
            open.pop_back();
            if (open.empty()) root_closed = true;
            i = j + 1;
            continue;
        }
        // start tag
        if (open.empty() && root_closed) return tags;                                  // junk after the document element
        XmlStartTag tag;
        const size_t nl = name_at(src, i + 1, &tag.name);
        if (!nl) return tags;
        size_t j = i + 1 + nl;
        bool self_closing = false, ok = false;
        while (j < n) {
            const size_t before = j;
            while (j < n && is_xml_space(data[j])) j++;
            if (j >= n) break;
            if (data[j] == '>') { ok = true; j++; break; }
            if (data[j] == '/') { if (j + 1 < n && data[j + 1] == '>') { ok = true; self_closing = true; j += 2; } break; }
            if (j == before) break;                                                     // attributes are separated by white space
            std::string an, av;
            const size_t al = name_at(src, j, &an);
            if (!al) break;
            j += al;
            while (j < n && is_xml_space(data[j])) j++;
            if (j >= n || data[j] != '=') break;
            j++;
            while (j < n && is_xml_space(data[j])) j++;
            if (j >= n || (data[j] != '"' && data[j] != '\'')) break;
            const unsigned char q = data[j++];
            bool closed = false;
            while (j < n) {
                if (data[j] == q) { closed = true; j++; break; }
                uint32_t cp;
                const int len = src.at(j, &cp);
                if (!len || cp == '<') break;
                if (cp == '&') { const size_t r = reference_at(src, j, &av); if (!r) break; j += r; continue; }
                if (cp == '\t' || cp == '\n' || cp == '\r') av += ' '; else append_utf8(av, cp);   // attribute-value normalisation
                j += len;
            }
            if (!closed) break;
            bool dup = false;
            for (auto& a : tag.attrs) dup |= a.first == an;
            if (dup) break;
            tag.attrs.emplace_back(std::move(an), std::move(av));
        }
        if (!ok) return tags;
        if (!self_closing) open.push_back(tag.name);
        else if (open.empty()) root_closed = true;
        tags.push_back(std::move(tag));
        i = j;
    }
    return tags;
}

// <Definition .../> attributes (attribute_parsers table, src/input_wav.c:334-342, handler :345-408)
void apply_definition_attr(const std::string& name, const std::string& value, iqgpu_wav_info* m)
{
    if (name == "SoftwareName") { copy_text(m->software_name, sizeof(m->software_name), value); m->software_name_present = 1; }
    else if (name == "SoftwareVersion") { copy_text(m->software_version, sizeof(m->software_version), value); m->software_version_present = 1; }
    else if (name == "RadioModel") { copy_text(m->radio_model, sizeof(m->radio_model), value); m->radio_model_present = 1; }
    else if (name == "RadioCenterFreq") {
        errno = 0;
        char* end = nullptr;
        const double v = strtod(value.c_str(), &end);
        if (errno == 0 && *end == '\0' && std::isfinite(v)) { m->center_freq_hz = v; m->center_freq_hz_present = 1; }
    } else if (name == "UTCSeconds") {
        if (!m->timestamp_unix_present) {
            errno = 0;
            char* end = nullptr;
            const long long v = strtoll(value.c_str(), &end, 10);
            if (errno == 0 && *end == '\0') { m->timestamp_unix = (int64_t)v; m->timestamp_unix_present = 1; }
        }
    } else if (name == "CurrentTimeUTC") {
        copy_text(m->timestamp_str, sizeof(m->timestamp_str), value);
        m->timestamp_str_present = 1;
        int day, month, year, hour, min, sec;       // SDR Console writes dd-mm-yyyy hh:mm:ss
        int64_t ts;
        if (sscanf(value.c_str(), "%d-%d-%d %d:%d:%d", &day, &month, &year, &hour, &min, &sec) == 6 &&
            utc_seconds(year, month, day, hour, min, sec, &ts)) {
            m->timestamp_unix = ts;
            m->timestamp_unix_present = 1;
        }
    }
}

bool parse_auxi_xml(const unsigned char* d, size_t n, iqgpu_wav_info* m)
{
    if (!d || !n) return false;
    for (const XmlStartTag& t : scan_xml_start_tags(d, n)) {
        if (t.name != "Definition") continue;
        for (const auto& a : t.attrs) apply_definition_attr(a.first, a.second, m);
    }
    const bool any = m->software_name_present || m->radio_model_present || m->center_freq_hz_present || m->timestamp_unix_present;
    if (any && m->software_name_present && strstr(m->software_name, "SDR Console")) m->source_software = IQGPU_SDR_CONSOLE;
    return any;
}

// SDRuno / SDR# binary auxi: SYSTEMTIME start (16 B), SYSTEMTIME stop (16 B), uint32 centre frequency at byte 32
// (src/input_wav.c:294-332)
bool parse_auxi_binary(const unsigned char* d, size_t n, iqgpu_wav_info* m)
{
    if (!d || n < 16 + 16 + 4) return false;
    bool got_time = false, got_freq = false;
    const unsigned year = le16(d), month = le16(d + 2), day = le16(d + 6), hour = le16(d + 8), min = le16(d + 10), sec = le16(d + 12);
    int64_t ts;
    if (utc_seconds((int)year, (int)month, (int)day, (int)hour, (int)min, (int)sec, &ts) && !m->timestamp_unix_present) {
        m->timestamp_unix = ts;
        m->timestamp_unix_present = 1;
        got_time = true;
        if (!m->timestamp_str_present) {
            snprintf(m->timestamp_str, sizeof(m->timestamp_str), "%04u-%02u-%02u %02u:%02u:%02u UTC", year, month, day, hour, min, sec);
            m->timestamp_str_present = 1;
        }
    }
    const uint32_t f = le32(d + 32);
    if (f > 0 && !m->center_freq_hz_present) {
        m->center_freq_hz = (double)f;
        m->center_freq_hz_present = 1;
        got_freq = true;
    }
    return got_time || got_freq;
}

// SDR# style names: ..._<centre>Hz... and ..._YYYYMMDD_HHMMSSZ... (src/input_wav.c:190-271)
bool parse_filename(const char* base, iqgpu_wav_info* m)
{
    if (!base) return false;
    bool something = false, looks_like_sdrsharp = false;
    const size_t len = strlen(base);

    if (!m->center_freq_hz_present) {
        // first "hz" in any letter case; the number runs from the last '_' in front of it up to it
        size_t hz = len;
        for (size_t i = 0; i + 1 < len; i++)
            if ((base[i] == 'H' || base[i] == 'h') && (base[i + 1] == 'Z' || base[i + 1] == 'z')) { hz = i; break; }
        if (hz < len) {
            size_t us = len;
            for (size_t i = 0; i < hz; i++)
                if (base[i] == '_') us = i;
            if (us < len && us + 1 < hz && hz - (us + 1) < 32) {
                const std::string num(base + us + 1, hz - (us + 1));
                char* end = nullptr;
                const double f = strtod(num.c_str(), &end);
                if (*end == '\0' && std::isfinite(f) && f > 0) {
                    m->center_freq_hz = f;
                    m->center_freq_hz_present = 1;
                    something = looks_like_sdrsharp = true;
                }
            }
        }
    }

    if (!m->timestamp_unix_present) {
        for (const char* p = strchr(base, '_'); p; p = strchr(p + 1, '_')) {
            // "_YYYYMMDD_HHMMSSZ": '_' at 9, 'Z' at 16
            if (strlen(p) < 17 || p[9] != '_' || p[16] != 'Z') continue;
            int year, month, day, hour, min, sec;
            if (sscanf(p, "_%4d%2d%2d_%2d%2d%2dZ", &year, &month, &day, &hour, &min, &sec) != 6) continue;
            int64_t ts;
            if (!utc_seconds(year, month, day, hour, min, sec, &ts)) continue;
            m->timestamp_unix = ts;
            m->timestamp_unix_present = 1;
            if (!m->timestamp_str_present) {
                snprintf(m->timestamp_str, sizeof(m->timestamp_str), "%04d-%02d-%02d %02d:%02d:%02d UTC", year, month, day, hour, min, sec);
                m->timestamp_str_present = 1;
            }
            something = looks_like_sdrsharp = true;
            break;
        }
    }

    if (m->source_software == IQGPU_SDR_SOFTWARE_UNKNOWN) {
        const char* label = nullptr;
        if (looks_like_sdrsharp) { m->source_software = IQGPU_SDR_SHARP; label = "SDR#"; }
        else if (strncmp(base, "SDRuno_", 7) == 0) { m->source_software = IQGPU_SDR_UNO; label = "SDRuno"; }
        else if (strncmp(base, "SDRconnect_", 11) == 0) { m->source_software = IQGPU_SDR_CONNECT; label = "SDRconnect"; }
        if (label && !m->software_name_present) {
            copy_text(m->software_name, sizeof(m->software_name), label);
            m->software_name_present = 1;
            something = true;
        }
    }
    return something;
}

const char* base_name(const char* path)
{
    const char* s = strrchr(path, '/');
    return s ? s + 1 : path;
}

// ---- RIFF / RF64 chunk walk (what sf_open does for a WAV file, as far as the reference depends on it) ----------------
int fail(const std::string& msg) { iqio::set_last_error(msg); return IQGPU_EINVAL; }

int probe_stream(FILE* f, const char* path, iqgpu_wav_info* info)
{
    memset(info, 0, sizeof(*info));
    if (fseeko(f, 0, SEEK_END) != 0) return fail(std::string("cannot seek in ") + path);
    const uint64_t file_len = (uint64_t)ftello(f);
    rewind(f);
    unsigned char hdr[12];
    if (fread(hdr, 1, 12, f) != 12) return fail(std::string("Error opening input file: ") + path + " is too short to be a WAV file");
    const bool rf64 = memcmp(hdr, "RF64", 4) == 0 || memcmp(hdr, "BW64", 4) == 0;
    if ((!rf64 && memcmp(hdr, "RIFF", 4) != 0) || memcmp(hdr + 8, "WAVE", 4) != 0)
        return fail(std::string("Error opening input file: ") + path + " is not a RIFF/RF64 WAVE file");
    info->container = rf64 ? IQGPU_CONTAINER_RF64 : IQGPU_CONTAINER_WAV;
    const uint32_t riff_size = le32(hdr + 4);

    bool have_fmt = false, have_data = false, have_ds64 = false, auxi_seen = false, auxi_ok = false;
    uint64_t ds64_data = 0;
    uint32_t block_align = 0;
    uint64_t pos = 12;
    while (pos + 8 <= file_len) {
        unsigned char ch[8];
        if (fseeko(f, (off_t)pos, SEEK_SET) != 0 || fread(ch, 1, 8, f) != 8) break;
        uint64_t size = le32(ch + 4);
        const uint64_t body = pos + 8;
        if (memcmp(ch, "ds64", 4) == 0 && size >= 24 && body + 24 <= file_len) {
            unsigned char b[24];
            if (fread(b, 1, 24, f) != 24) break;
            ds64_data = le64(b + 8);
            have_ds64 = true;
        } else if (memcmp(ch, "fmt ", 4) == 0 && !have_fmt) {
            unsigned char b[40];
            const size_t want = size < 40 ? (size_t)size : 40;
            if (size < 16 || fread(b, 1, want, f) != want) return fail(std::string("Error opening input file: ") + path + " has a truncated fmt chunk");
            info->format_tag = le16(b);
            info->channels = le16(b + 2);
            info->sample_rate_hz = (int32_t)le32(b + 4);
            block_align = le16(b + 12);
            info->bits_per_sample = le16(b + 14);
            if (info->format_tag == 0xFFFE && want >= 26) info->format_tag = le16(b + 24);   // WAVE_FORMAT_EXTENSIBLE: first word of the sub-format GUID
            have_fmt = true;
        } else if (memcmp(ch, "data", 4) == 0 && !have_data) {
            if (!have_fmt) return fail(std::string("Error opening input file: ") + path + " has its data chunk in front of the fmt chunk");
            if (rf64 && size == 0xFFFFFFFFu && have_ds64) size = ds64_data;
            // a recorder that was stopped hard leaves 0 (or all ones) here: the payload then runs to the end of the file
            if (size > file_len - body || size == 0xFFFFFFFFu || (size == 0 && (riff_size == 0 || riff_size == 0xFFFFFFFFu || riff_size == 36) && file_len > body))
                size = file_len - body;
            info->data_offset = body;
            info->data_bytes = size;
            have_data = true;
        } else if (memcmp(ch, "auxi", 4) == 0 && !auxi_seen) {
            // process_specific_chunk (src/input_wav.c:146-182): the first auxi chunk only, 1 byte .. 1 MiB
            auxi_seen = true;
            if (size > 0 && size <= kMaxMetadataChunk && body + size <= file_len) {
                std::vector<unsigned char> buf((size_t)size);
                if (fread(buf.data(), 1, buf.size(), f) == buf.size()) auxi_ok = iqgpu_wav_parse_auxi(buf.data(), buf.size(), info) != 0;
            }
        }
        pos = body + size + (size & 1);                                                 // chunks are word aligned
    }
    if (!have_fmt || !have_data) return fail(std::string("Error opening input file: ") + path + " has no " + (have_fmt ? "data" : "fmt") + " chunk");

    // wav_initialize's checks, in its order (src/input_wav.c:567-598)
    if (info->channels != 2)
        return fail("Error: Input file must have 2 channels (I/Q), but found " + std::to_string(info->channels) + ".");
    if (info->format_tag == 1 && info->bits_per_sample == 16) info->sample_format = IQGPU_FMT_CS16;
    else if (info->format_tag == 1 && info->bits_per_sample == 8) info->sample_format = IQGPU_FMT_CU8;
    else {
        char msg[256];
        snprintf(msg, sizeof(msg), "Error: Input WAV file uses an unsupported PCM subtype (format tag %d, %d bits). "
                 "Supported WAV PCM subtypes are 16-bit Signed (cs16) and 8-bit Unsigned (cu8).", info->format_tag, info->bits_per_sample);
        return fail(msg);
    }
    if (info->sample_rate_hz <= 0) return fail("Error: Invalid input sample rate (" + std::to_string(info->sample_rate_hz) + " Hz).");
    const uint32_t frame_bytes = (uint32_t)info->channels * (uint32_t)(info->bits_per_sample / 8);
    (void)block_align;                                                                 // libsndfile derives the block width the same way for PCM
    info->frames = info->data_bytes / frame_bytes;
    info->data_bytes = info->frames * frame_bytes;                                      // sf_read_raw stops at the last whole frame

    const bool from_name = iqgpu_wav_parse_filename(base_name(path), info) != 0;
    info->metadata_present = (auxi_ok || from_name) ? 1 : 0;
    return IQGPU_OK;
}

}  // namespace

extern "C" {

int iqgpu_wav_parse_auxi(const void* chunk, size_t bytes, iqgpu_wav_info* info)
{
    if (!chunk || !info) return 0;
    const unsigned char* d = (const unsigned char*)chunk;
    if (parse_auxi_xml(d, bytes, info)) return 1;
    return parse_auxi_binary(d, bytes, info) ? 1 : 0;
}

int iqgpu_wav_parse_filename(const char* base_filename, iqgpu_wav_info* info)
{
    if (!base_filename || !info) return 0;
    return parse_filename(base_filename, info) ? 1 : 0;
}

int iqgpu_wav_probe(const char* path, iqgpu_wav_info* info)
{
    if (!path || !info) return fail("null argument");
    FILE* f = fopen(path, "rb");
    if (!f) return fail(std::string("Error opening input file: ") + path);
    const int rc = probe_stream(f, path, info);
    fclose(f);
    return rc;
}

int iqgpu_wav_center_target_shift(const iqgpu_wav_info* info, float center_target_hz, double freq_shift_hz_arg, double* nco_shift_hz)
{
    if (!info || !nco_shift_hz) return fail("null argument");
    if (center_target_hz == 0.0f) { *nco_shift_hz = freq_shift_hz_arg; return IQGPU_OK; }
    if (freq_shift_hz_arg != 0.0)
        return fail("Conflicting frequency shift options provided. Cannot use --freq-shift and --wav-center-target-freq at the same time.");
    if (!info->center_freq_hz_present)
        return fail("Option --wav-center-target-freq was used, but the input WAV file does not contain the required center frequency metadata.");
    *nco_shift_hz = info->center_freq_hz - (double)center_target_hz;
    return IQGPU_OK;
}

size_t iqgpu_wav_header_bytes(int container)
{
    return container == IQGPU_CONTAINER_WAV ? 44 : container == IQGPU_CONTAINER_RF64 ? 80 : 0;
}

int iqgpu_wav_build_header(int container, int output_format, int sample_rate_hz, uint64_t data_bytes, void* header, size_t capacity)
{
    const size_t n = iqgpu_wav_header_bytes(container);
    if (!n) return fail("not a WAV or RF64 container");
    if (!header || capacity < n) { iqio::set_last_error("header buffer too small"); return IQGPU_ECAPACITY; }
    if (output_format != IQGPU_FMT_CS16 && output_format != IQGPU_FMT_CU8)
        return fail("Invalid sample format for WAV/RF64 container. Only 'cs16' and 'cu8' are supported.");
    if (sample_rate_hz <= 0) return fail("libsndfile does not support the requested format (sample rate <= 0)");
    const uint32_t bytes = output_format == IQGPU_FMT_CS16 ? 2 : 1, frame = 2 * bytes;
    unsigned char* h = (unsigned char*)header;
    unsigned char fmt[16];
    put16(fmt, 1);                      // WAVE_FORMAT_PCM
    put16(fmt + 2, 2);                  // I, Q
    put32(fmt + 4, (uint32_t)sample_rate_hz);
    put32(fmt + 8, (uint32_t)sample_rate_hz * frame);
    put16(fmt + 12, frame);
    put16(fmt + 14, 8 * bytes);
    if (container == IQGPU_CONTAINER_WAV) {
        // sizes past 32 bits cannot be told: all ones, which readers take as "to the end of the file"
        const bool fits = data_bytes <= 0xFFFFFFFFull - 36;
        memcpy(h, "RIFF", 4); put32(h + 4, fits ? (uint32_t)(data_bytes + 36) : 0xFFFFFFFFu); memcpy(h + 8, "WAVE", 4);
        memcpy(h + 12, "fmt ", 4); put32(h + 16, 16); memcpy(h + 20, fmt, 16);
        memcpy(h + 36, "data", 4); put32(h + 40, fits ? (uint32_t)data_bytes : 0xFFFFFFFFu);
    } else {
        memcpy(h, "RF64", 4); put32(h + 4, 0xFFFFFFFFu); memcpy(h + 8, "WAVE", 4);
        memcpy(h + 12, "ds64", 4); put32(h + 16, 28);
        put64(h + 20, data_bytes + 72);                 // RIFF size: the file without the first 8 bytes
        put64(h + 28, data_bytes);
        put64(h + 36, data_bytes / frame);              // sample (frame) count
        put32(h + 44, 0);                               // no chunk-size table
        memcpy(h + 48, "fmt ", 4); put32(h + 52, 16); memcpy(h + 56, fmt, 16);
        memcpy(h + 72, "data", 4); put32(h + 76, 0xFFFFFFFFu);
    }
    return IQGPU_OK;
}

int iqgpu_wavfile_run(const iqgpu_chain_config* cfg, int device, const char* in_path, int in_container, const char* out_path,
                      int out_container, float center_target_hz, size_t train_chunks, iqgpu_rawfile_stats* stats, iqgpu_wav_info* in_info)
{
    return iqio::wavfile_run(cfg, 1, device, in_path, in_container, &out_path, &out_container, &center_target_hz, train_chunks,
                             stats, in_info, iqio::process_one);
}

}  // extern "C"

int iqio::wavfile_run(const iqgpu_chain_config* cfgs_in, size_t n, int device, const char* in_path, int in_container,
                      const char* const* out_paths, const int* out_containers, const float* center_target_hz, size_t train_chunks,
                      iqgpu_rawfile_stats* stats, iqgpu_wav_info* in_info, ProcessFn process)
{
    if (!cfgs_in || !in_path || !out_paths || !out_containers) return fail("null argument");
    if (n == 0) return fail("n_channels must be at least 1");
    if (in_container < IQGPU_CONTAINER_RAW || in_container > IQGPU_CONTAINER_RF64) return fail("unknown container");
    for (size_t k = 0; k < n; k++) {
        if (!out_paths[k]) return fail(channel_prefix(k, n) + "null argument");
        if (out_containers[k] < IQGPU_CONTAINER_RAW || out_containers[k] > IQGPU_CONTAINER_RF64) return fail(channel_prefix(k, n) + "unknown container");
    }
    if (stats) memset(stats, 0, n * sizeof(*stats));
    if (in_info) memset(in_info, 0, sizeof(*in_info));
    std::vector<iqgpu_chain_config> cfgs(cfgs_in, cfgs_in + n);
    auto target = [&](size_t k) { return center_target_hz ? center_target_hz[k] : 0.0f; };

    FILE* fin = fopen(in_path, "rb");
    if (!fin) return fail(std::string("Error opening input file: ") + in_path);
    uint64_t in_limit = UINT64_MAX;
    if (in_container != IQGPU_CONTAINER_RAW) {
        iqgpu_wav_info wi;
        int rc = probe_stream(fin, in_path, &wi);
        for (size_t k = 0; k < n && !rc; k++) {
            rc = iqgpu_wav_center_target_shift(&wi, target(k), cfgs[k].freq_shift_hz, &cfgs[k].freq_shift_hz);
            if (rc && n > 1) iqio::set_last_error(channel_prefix(k, n) + iqgpu_rawfile_last_error());
        }
        if (in_info) *in_info = wi;
        if (rc) { fclose(fin); return rc; }
        for (auto& cfg : cfgs) {
            cfg.input_format = wi.sample_format;                // src/input_wav.c:575-577
            cfg.input_rate_hz = (double)wi.sample_rate_hz;      // :597
        }
        in_limit = wi.data_bytes;
        if (fseeko(fin, (off_t)wi.data_offset, SEEK_SET) != 0) { fclose(fin); return fail(std::string("cannot seek in ") + in_path); }
    } else {
        for (size_t k = 0; k < n; k++)
            if (target(k) != 0.0f) { fclose(fin); return fail(channel_prefix(k, n) + "Option --wav-center-target-freq needs a WAV input"); }
    }
    // output side: wav_common_validate_options + wav_common_initialize (src/output_wav_common.c:46-118), one header per channel
    std::vector<unsigned char> headers(80 * n);
    std::vector<size_t> header_bytes(n);
    for (size_t k = 0; k < n; k++) {
        iqgpu_chain_config& cfg = cfgs[k];
        // setup.c:99: with --no-resample the target rate IS the source rate (known only now for a WAV input)
        if (cfg.no_resample) cfg.target_rate_hz = (double)(int)cfg.input_rate_hz;
        header_bytes[k] = iqgpu_wav_header_bytes(out_containers[k]);
        if (header_bytes[k]) {
            const int rc = iqgpu_wav_build_header(out_containers[k], cfg.output_format, (int)cfg.target_rate_hz, 0, &headers[80 * k], 80);
            if (rc) {
                if (n > 1) iqio::set_last_error(channel_prefix(k, n) + iqgpu_rawfile_last_error());
                fclose(fin);
                return rc;
            }
        }
    }

    Channels ch;
    ch.process = process;
    std::string err;
    int rc = ch.open(cfgs.data(), n, device, out_paths, "Error opening output WAV file ", err);
    if (rc) { fclose(fin); iqio::set_last_error(err); return rc; }
    std::vector<iqgpu_rawfile_stats> st(n);
    memset(st.data(), 0, n * sizeof(st[0]));
    for (size_t k = 0; k < n && !rc; k++)
        if (header_bytes[k] && fwrite(&headers[80 * k], 1, header_bytes[k], ch.fouts[k]) != header_bytes[k]) {
            rc = IQGPU_EINVAL;
            err = channel_prefix(k, n) + "write error on the output file";
        }
    if (!rc) rc = iqio::run_stream(ch, cfgs.data(), fin, in_limit, train_chunks, st.data(), err);
    for (size_t k = 0; k < n && !rc; k++) {
        if (!header_bytes[k]) continue;
        // what sf_close does: the sizes now that they are known
        iqgpu_wav_build_header(out_containers[k], cfgs[k].output_format, (int)cfgs[k].target_rate_hz, st[k].bytes_written, &headers[80 * k], 80);
        if (fseeko(ch.fouts[k], 0, SEEK_SET) != 0 || fwrite(&headers[80 * k], 1, header_bytes[k], ch.fouts[k]) != header_bytes[k]) {
            rc = IQGPU_EINVAL;
            err = channel_prefix(k, n) + "cannot finalise the output header";
        }
    }
    const int rc_close = ch.close(err);
    if (!rc) rc = rc_close;
    fclose(fin);
    if (stats) memcpy(stats, st.data(), n * sizeof(st[0]));
    if (rc) iqio::set_last_error(err);
    return rc;
}
