// graph_front.cu -- front end of the generated cproc graphs (SURVEY 8 f-1).
//
//  * cproc_cuda_graph_parse: reads the C text that epid_cproc.erl generates -- the wire
//    format between the Erlang side and the C side of the reference
//    (linux/test_cproc.c:11-17, stm32f103/bp5_plugin.c:1-9):
//        #define CPROC_NB_INPUTS 1
//        void cproc_update(w *input, w g) {
//            PROC_COND(g&0b1, n1, edge, NULL, NULL, .in = input[0]);
//            PROC_COND(g&0b1, n2, acc,  NULL, NULL, .in = n1.out);
//            cproc_output(2, n2.out);
//        }
//    into the node table of CPROC_CUDA_GRAPH (one row per PROC_COND / PROC statement,
//    generic/cproc.h:72-81).
//  * graph JIT: a graph is straight-line code over its node states, so the renderer
//    generates CUDA source for exactly this graph (every node state word a named
//    register, every source a literal register name, masks as immediates) and compiles
//    it with NVRTC for sm_100a when the batch is created.  PLANAR streams are staged
//    with tensor TMA as in pbulk::k_planar_tma; INTERLEAVED streams are read in
//    16-frame batches.  libnvrtc is loaded with dlopen: without it (or with graph_jit=0)
//    graphs of up to 16 nodes run on the table-driven kernel of k_graph.cu.
#include "common.cuh"
#include <ctype.h>
#include <dlfcn.h>
#include <regex>
#include <unordered_map>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

// ---------------------------------------------------------------------------
// parser

namespace {

struct Cursor {
    const char *p;
    std::string err;
    void ws() { while (*p && isspace((unsigned char)*p)) ++p; }
    bool lit(const char *s) { ws(); size_t n = strlen(s); if (strncmp(p, s, n) == 0) { p += n; return true; } return false; }
    bool ident(std::string *out) {
        ws();
        if (!(isalpha((unsigned char)*p) || *p == '_')) return false;
        const char *b = p;
        while (isalnum((unsigned char)*p) || *p == '_') ++p;
        out->assign(b, p);
        return true;
    }
    bool number(uint64_t *out) {                       // decimal, 0x.., 0b.. (gcc extension used by the generator)
        ws();
        if (!isdigit((unsigned char)*p)) return false;
        uint64_t v = 0;
        if (p[0] == '0' && (p[1] == 'b' || p[1] == 'B')) {
            p += 2;
            if (*p != '0' && *p != '1') return false;
            while (*p == '0' || *p == '1') v = (v << 1) | (uint64_t)(*p++ - '0');
        } else if (p[0] == '0' && (p[1] == 'x' || p[1] == 'X')) {
            p += 2;
            if (!isxdigit((unsigned char)*p)) return false;
            while (isxdigit((unsigned char)*p)) { const char c = *p++; v = (v << 4) | (uint64_t)(isdigit((unsigned char)c) ? c - '0' : (tolower(c) - 'a' + 10)); }
        } else {
            while (isdigit((unsigned char)*p)) v = v * 10 + (uint64_t)(*p++ - '0');
        }
        while (*p == 'u' || *p == 'U' || *p == 'l' || *p == 'L') ++p;
        *out = v;
        return true;
    }
};

std::string strip_comments(const char *s) {
    std::string o;
    while (*s) {
        if (s[0] == '/' && s[1] == '/') { while (*s && *s != '\n') ++s; }
        else if (s[0] == '/' && s[1] == '*') { s += 2; while (*s && !(s[0] == '*' && s[1] == '/')) ++s; if (*s) s += 2; o += ' '; }
        else o += *s++;
    }
    return o;
}

// top-level comma split of a parenthesised argument list starting after '('; leaves c.p after ')'
bool split_args(Cursor &c, std::vector<std::string> *args) {
    int depth = 1;
    std::string cur;
    while (*c.p) {
        const char ch = *c.p++;
        if (ch == '(' || ch == '[' || ch == '{') ++depth;
        if (ch == ')' || ch == ']' || ch == '}') { if (--depth == 0) { args->push_back(cur); return true; } }
        if (ch == ',' && depth == 1) { args->push_back(cur); cur.clear(); continue; }
        cur += ch;
    }
    return false;
}

std::string trim(const std::string &s) {
    size_t a = 0, b = s.size();
    while (a < b && isspace((unsigned char)s[a])) ++a;
    while (b > a && isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

// condition of a PROC_COND: `g & MASK`, `MASK & g`, a constant, optionally parenthesised
bool parse_cond(std::string s, uint32_t *mask, std::string *why) {
    s = trim(s);
    while (s.size() >= 2 && s.front() == '(' && s.back() == ')') s = trim(s.substr(1, s.size() - 2));
    Cursor c{s.c_str(), ""};
    std::string id; uint64_t v = 0;
    if (c.number(&v)) {
        c.ws();
        if (*c.p == 0) { *mask = v ? 0xFFFFFFFFu : 0u; return true; }          // PROC(...) == PROC_COND(1, ...)
        if (*c.p == '&') { ++c.p; if (c.ident(&id)) { c.ws(); if (*c.p == 0) { *mask = (uint32_t)v; return true; } } }
    } else if (c.ident(&id)) {
        c.ws();
        if (*c.p == '&') { ++c.p; if (c.number(&v)) { c.ws(); if (*c.p == 0) { *mask = (uint32_t)v; return true; } } }
    }
    *why = "condition '" + s + "' is not of the form <changed> & <mask>";
    return false;
}

}  // namespace

extern "C" int cproc_cuda_graph_parse(const char *text, cproc_cuda_node *nodes, uint32_t max_nodes, cproc_cuda_graph_info *info) {
    if (!text || !nodes || !info) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: NULL argument");
    memset(info, 0, sizeof(*info));
    const std::string src = strip_comments(text);
    std::vector<std::string> names;
    uint32_t max_input = 0; bool any_input = false;
    uint32_t n_out = 0, n_param_words = 0;
    bool have_define = false;
    // #define CPROC_NB_INPUTS n
    {
        const char *d = strstr(src.c_str(), "CPROC_NB_INPUTS");
        while (d) {
            const char *ls = d; while (ls > src.c_str() && ls[-1] != '\n') --ls;
            Cursor c{ls, ""};
            if (c.lit("#") && c.lit("define") && c.lit("CPROC_NB_INPUTS")) { uint64_t v; if (c.number(&v)) { info->n_inputs = (uint32_t)v; have_define = true; break; } }
            d = strstr(d + 1, "CPROC_NB_INPUTS");
        }
    }
    const char *p = src.c_str();
    while (*p) {
        if (!(isalpha((unsigned char)*p) || *p == '_')) { ++p; continue; }
        Cursor c{p, ""};
        std::string id;
        c.ident(&id);
        p = c.p;
        const bool is_cond = id == "PROC_COND", is_proc = id == "PROC", is_out_f = id == "cproc_output_f";
        if (!is_cond && !is_proc && id != "cproc_output" && !is_out_f) continue;
        c.ws();
        if (*c.p != '(') continue;                      // e.g. the definition `static inline void cproc_output(`... has '(' too, handled below
        ++c.p;
        std::vector<std::string> a;
        if (!split_args(c, &a)) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: unbalanced parentheses after %s", id.c_str());
        p = c.p;
        if (id == "cproc_output" || is_out_f) {
            // a call has two expression arguments; the definition `cproc_output(uint32_t index, w value)` is skipped
            if (a.size() != 2) continue;
            Cursor n{a[0].c_str(), ""}; uint64_t idx;
            if (!n.number(&idx)) continue;
            std::string e = trim(a[1]);
            const size_t dot = e.find('.');
            if (dot == std::string::npos || trim(e.substr(dot + 1)) != "out")
                return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: cproc_output value '%s' is not <node>.out", e.c_str());
            const std::string nm = trim(e.substr(0, dot));
            size_t k = 0;
            while (k < names.size() && names[k] != nm) ++k;
            if (k == names.size()) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: cproc_output reads unknown node '%s'", nm.c_str());
            if (n_out >= CPROC_CUDA_GRAPH_MAX_OUTPUTS) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: more than %d cproc_output statements", CPROC_CUDA_GRAPH_MAX_OUTPUTS);
            if (cproc_kind_out_float(nodes[k].type) != is_out_f)
                return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: '%s.out' is a %s: use %s", nm.c_str(), is_out_f ? "w" : "float", is_out_f ? "cproc_output" : "cproc_output_f (cproc_output would convert the value)");
            if (is_out_f) info->out_is_float |= 1u << n_out;
            info->out_nodes[n_out] = (uint32_t)k; info->out_indices[n_out] = (uint32_t)idx;
            if (n_out++ == 0) { info->out_node = (uint32_t)k; info->out_index = (uint32_t)idx; }
            continue;
        }
        const size_t base = is_cond ? 1 : 0;             // PROC(inst, type, cfg, prm, inits...)
        if (a.size() < base + 4) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: %s needs an instance, a type, config, param and the inputs", id.c_str());
        cproc_cuda_node nd;
        std::string why;
        if (is_cond) { if (!parse_cond(a[0], &nd.cond_mask, &why)) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: %s", why.c_str()); }
        else nd.cond_mask = 0xFFFFFFFFu;
        const std::string inst = trim(a[base]), type = trim(a[base + 1]), cfg = trim(a[base + 2]), prm = trim(a[base + 3]);
        bool cfg_null = cfg == "NULL" || cfg == "0";
        nd.src = nd.src2 = CPROC_CUDA_SRC_ZERO;
        uint32_t n_in_expected = 1;
        uint32_t kind = CPROC_CUDA_NODE_KINDS;
        for (uint32_t q = 0; q < CPROC_CUDA_NODE_KINDS; ++q) if (q != CPROC_CUDA_NODE_PDM && type == k_cproc_kinds[q].name) kind = q;
        if (kind == CPROC_CUDA_NODE_GLIDE || kind == CPROC_CUDA_NODE_GLIDE_F) {
            // const glide_config: &(glide_config){ .div_log = L }  (any spelling that names div_log = <number>)
            const size_t f = cfg.find("div_log");
            uint64_t L = 0;
            bool ok = f != std::string::npos;
            if (ok) { Cursor q{cfg.c_str() + f + 7, ""}; ok = q.lit("=") && q.number(&L) && L >= 1 && L <= 24; }
            if (!ok) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': %s needs a config with .div_log = 1..24", inst.c_str(), type.c_str());
            nd.type = kind | ((uint32_t)L << 8);
            cfg_null = true;
        }
        else if (type.size() == 4 && type.compare(0, 3, "pdm") == 0 && type[3] >= '1' && type[3] <= '4') {
            // pdmK_update(&s, in, out_shift, dither), pdm.h:13-77: &(pdm_config){ .out_shift = S }
            const size_t f = cfg.find("out_shift");
            uint64_t S = 0;
            bool ok = f != std::string::npos;
            if (ok) { Cursor q{cfg.c_str() + f + 9, ""}; ok = q.lit("=") && q.number(&S) && S <= 31; }
            if (!ok) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': %s needs a config with .out_shift = 0..31", inst.c_str(), type.c_str());
            kind = CPROC_CUDA_NODE_PDM;
            nd.type = CPROC_CUDA_NODE_PDM_K(type[3] - '0', S);
            cfg_null = true;
            n_in_expected = type[3] == '1' ? 1 : 2;             // pdm1 takes no dither (pdm.h:13)
        }
        else if (kind < CPROC_CUDA_NODE_KINDS) nd.type = kind;
        else return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s' has unknown processor type '%s' (acc, edge, glide, pdm1..pdm4, phasor_f, svf, env, onepole, gain, asfloat, glide_f, mul)", inst.c_str(), type.c_str());
        const cproc_kind_meta &meta = k_cproc_kinds[kind];
        const bool ext = kind > CPROC_CUDA_NODE_PDM;
        if (!cfg_null || (meta.n_param == 0 && prm != "NULL" && prm != "0"))
            return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': %s has empty config and param records, expected NULL", inst.c_str(), type.c_str());
        if (meta.n_param) {
            // NAME_param: `&<identifier>` (uploaded by the host) or `&(NAME_param){ .field = <number>, ... }`
            if (n_param_words + meta.n_param > CPROC_CUDA_GRAPH_MAX_PARAM_WORDS) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: param record exceeds %d words", CPROC_CUDA_GRAPH_MAX_PARAM_WORDS);
            // a compound literal with several members needs parentheses around it to survive the preprocessor's argument split
            std::string pe = prm;
            while (pe.size() >= 2 && pe.front() == '(' && pe.back() == ')') {
                int depth = 0; bool outer = true;
                for (size_t z = 0; z + 1 < pe.size(); ++z) { if (pe[z] == '(') ++depth; else if (pe[z] == ')') --depth; if (depth == 0) { outer = false; break; } }
                if (!outer) break;
                pe = trim(pe.substr(1, pe.size() - 2));
            }
            Cursor q{pe.c_str(), ""};
            if (!q.lit("&")) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': %s needs a param record (&<name> or &(%s_param){ ... })", inst.c_str(), type.c_str(), type.c_str());
            std::string id2;
            if (q.lit("(")) {
                if (!q.ident(&id2) || id2 != type + "_param" || !q.lit(")") || !q.lit("{"))
                    return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': expected &(%s_param){ ... }", inst.c_str(), type.c_str());
                while (true) {
                    q.ws();
                    if (q.lit("}")) break;
                    std::string f;
                    if (!q.lit(".") || !q.ident(&f) || !q.lit("=")) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': expected '.field = value' in the param initialiser", inst.c_str());
                    uint32_t fi = 0;
                    while (fi < meta.n_param && f != meta.param[fi]) ++fi;
                    if (fi == meta.n_param) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': %s_param has no member '%s'", inst.c_str(), type.c_str(), f.c_str());
                    q.ws();
                    char *end = nullptr;
                    uint32_t word;
                    if ((meta.param_f >> fi) & 1u) {
                        const float v = strtof(q.p, &end);
                        if (end == q.p) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': '%s' needs a number", inst.c_str(), f.c_str());
                        memcpy(&word, &v, 4);
                        while (*end == 'f' || *end == 'F') ++end;
                        q.p = end;
                    } else {
                        uint64_t v;
                        if (!q.number(&v)) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': '%s' needs an unsigned integer", inst.c_str(), f.c_str());
                        word = (uint32_t)v;
                    }
                    info->param_init[n_param_words + fi] = word;
                    q.lit(",");
                }
            } else if (!q.ident(&id2)) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': param expression not understood", inst.c_str());
            q.ws();
            if (*q.p) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': trailing text after the param expression", inst.c_str());
            n_param_words += meta.n_param;
        }
        for (const std::string &nm : names) if (nm == inst) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s' bound twice", inst.c_str());
        const bool is_pdm = kind == CPROC_CUDA_NODE_PDM;
        if ((!ext && a.size() < base + 5) || a.size() > base + 4 + meta.n_input)
            return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': %s has exactly %u input%s (.in%s)", inst.c_str(), type.c_str(), n_in_expected, n_in_expected > 1 ? "s" : "", is_pdm ? ", .dither" : "");
        // designated initialisers: .<input> = input[k] | <node>.out ; a member the statement does not name is 0 (C)
        bool have[2] = {false, false};
        for (size_t ai = base + 4; ai < a.size(); ++ai) {
            if (ext && trim(a[ai]).empty()) continue;            // PROC(n, phasor_f, NULL, &p) leaves the variadic part empty
            Cursor b{a[ai].c_str(), ""};
            std::string f;
            uint32_t fi = meta.n_input;
            if (b.lit(".") && b.ident(&f) && b.lit("=")) { fi = 0; while (fi < meta.n_input && f != meta.input[fi]) ++fi; }
            if (fi == meta.n_input) {
                if (ext) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': expected '.%s = ...'", inst.c_str(), meta.input[0]);
                return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': expected '.in = ...'%s", inst.c_str(), is_pdm ? " / '.dither = ...'" : "");
            }
            int32_t srcv = 0;
            std::string s0;
            if (!b.ident(&s0)) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': input expression not understood", inst.c_str());
            if (b.lit("[")) {
                uint64_t k;
                if (s0 != "input" || !b.number(&k) || !b.lit("]")) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': expected input[<k>]", inst.c_str());
                if (k >= 65536) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': input[%llu] is out of range", inst.c_str(), (unsigned long long)k);
                srcv = -(int32_t)k - 1;
                if (!any_input || k > max_input) max_input = (uint32_t)k;
                any_input = true;
            } else {
                std::string fo;
                if (!b.lit(".") || !b.ident(&fo) || fo != "out") return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': expected <node>.out", inst.c_str());
                size_t k = 0;
                while (k < names.size() && names[k] != s0) ++k;
                if (k == names.size()) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s' reads '%s', which is not bound yet (ANF)", inst.c_str(), s0.c_str());
                if (cproc_kind_out_float(nodes[k].type) && !((meta.input_f >> fi) & 1u))
                    return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': '%s.out' is a float and .%s is a w (the conversion is undefined in C for negative values)", inst.c_str(), s0.c_str(), f.c_str());
                srcv = (int32_t)k;
            }
            b.ws();
            if (*b.p) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': trailing text in the input expression", inst.c_str());
            if (have[fi]) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': .%s given twice", inst.c_str(), f.c_str());
            have[fi] = true;
            if (fi == 0) nd.src = srcv; else nd.src2 = srcv;
        }
        if (!ext && !have[0]) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': expected '.in = ...'", inst.c_str());
        if (is_pdm && !have[1]) {
            if (n_in_expected == 2) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: node '%s': %s needs '.dither = ...'", inst.c_str(), type.c_str());
            nd.src2 = nd.src;                                    // pdm1: unused, keep the row valid
        }
        if (meta.n_input < 2) nd.src2 = 0;                       // one-input processors: src2 is ignored
        if (names.size() >= max_nodes) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: more than %u nodes", max_nodes);
        nodes[names.size()] = nd;
        names.push_back(inst);
    }
    if (names.empty()) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: no PROC_COND / PROC statement found");
    if (n_out == 0) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: no cproc_output(index, node.out) statement found");
    info->n_outputs = n_out;
    info->n_param_words = n_param_words;
    const uint32_t need = any_input ? max_input + 1 : 0;
    if (!have_define) info->n_inputs = need;
    if (info->n_inputs < need) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_parse: input[%u] used but CPROC_NB_INPUTS is %u", max_input, info->n_inputs);
    info->n_nodes = (uint32_t)names.size();
    return 0;
}

// ---------------------------------------------------------------------------
// JIT

namespace {

typedef int (*nvrtcCreateProgram_t)(void **, const char *, const char *, int, const char *const *, const char *const *);
typedef int (*nvrtcCompileProgram_t)(void *, int, const char *const *);
typedef int (*nvrtcGetSize_t)(void *, size_t *);
typedef int (*nvrtcGetData_t)(void *, char *);
typedef int (*nvrtcDestroyProgram_t)(void **);

struct Nvrtc {
    void *h = nullptr;
    nvrtcCreateProgram_t create = nullptr;
    nvrtcCompileProgram_t compile = nullptr;
    nvrtcGetSize_t cubin_size = nullptr, log_size = nullptr;
    nvrtcGetData_t cubin = nullptr, log = nullptr;
    nvrtcDestroyProgram_t destroy = nullptr;
    bool tried = false;
};
Nvrtc g_nvrtc;

bool nvrtc_load() {
    if (g_nvrtc.tried) return g_nvrtc.h != nullptr;
    g_nvrtc.tried = true;
    const char *names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"};
    void *h = nullptr;
    for (const char *n : names) if ((h = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
    if (!h) {
        // the wheel layout: nvidia/cuda_nvrtc/lib next to torch (searched through the loaded process image)
        return false;
    }
    Nvrtc &r = g_nvrtc;
    r.create = (nvrtcCreateProgram_t)dlsym(h, "nvrtcCreateProgram");
    r.compile = (nvrtcCompileProgram_t)dlsym(h, "nvrtcCompileProgram");
    r.cubin_size = (nvrtcGetSize_t)dlsym(h, "nvrtcGetCUBINSize");
    r.cubin = (nvrtcGetData_t)dlsym(h, "nvrtcGetCUBIN");
    r.log_size = (nvrtcGetSize_t)dlsym(h, "nvrtcGetProgramLogSize");
    r.log = (nvrtcGetData_t)dlsym(h, "nvrtcGetProgramLog");
    r.destroy = (nvrtcDestroyProgram_t)dlsym(h, "nvrtcDestroyProgram");
    if (!r.create || !r.compile || !r.cubin_size || !r.cubin || !r.log_size || !r.log || !r.destroy) { dlclose(h); return false; }
    r.h = h;
    return true;
}

// The fixed part of the generated translation unit.  GRAPH_* macros and the two
// generated code blocks (GRAPH_DECL_STATE .. GRAPH_TICK) come first.
const char *k_jit_head = "typedef unsigned int uint32_t;\ntypedef unsigned long long uint64_t;\ntypedef int int32_t;\n";
const char *k_jit_tail = R"SRC(

struct GraphParams {                       // must match k_graph.cu
    uint32_t *st;
    uint64_t npad, n;
    const void *nodes;
    uint32_t n_nodes, n_inputs, out_node, state_words;
    const uint32_t *in;
    const uint32_t *changed;
    uint32_t *out;
    uint64_t F;
    uint32_t layout;
    uint32_t n_outputs;
    uint32_t out_nodes[16];
    const uint32_t *prm;
};

// one tick of one instance: x[] = this tick's inputs, g = changed mask; o[] = the output words (GRAPH_NOUT of them)
__device__ __forceinline__ void graph_tick(GState &S, const GParam &P, const uint32_t *x, uint32_t g, uint32_t *o) { GRAPH_TICK(x, g) GRAPH_OUTS(o) }
#define TICK(x, g, o) graph_tick(S, P, x, g, o)

// [F][n_inputs][inst] in, [F][inst] changed / out: coalesced as they are; 16-frame batches
// make the independent loads explicit (in may alias out).
#define GI_B (GRAPH_NIN + GRAPH_NOUT <= 3 ? 16 : 8)        // frames per batch: fewer when many streams are in flight
extern "C" __global__ void __launch_bounds__(128) graph_interleaved(const GraphParams p) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    GRAPH_DECL_STATE
    GRAPH_LOAD_STATE(p.st, p.npad, i)
    GParam P = {};
    GRAPH_LOAD_PARAM(p.prm, p.npad, i)
    const uint32_t *src = p.in + i;
    const uint32_t *chg = GRAPH_HAS_CHANGED ? p.changed + i : 0;
    uint32_t *dst = p.out + i;
    const uint64_t n = p.n;
    uint64_t t = 0;
    for (; t + GI_B <= p.F; t += GI_B) {
        uint32_t x[GI_B][GRAPH_NINA], g[GI_B], o[GI_B][GRAPH_NOUT];
#pragma unroll
        for (int k = 0; k < GI_B; ++k) {
#pragma unroll
            for (int j = 0; j < GRAPH_NIN; ++j) x[k][j] = __ldcs(src + ((t + k) * GRAPH_NIN + j) * n);
            g[k] = GRAPH_HAS_CHANGED ? __ldcs(chg + (t + k) * n) : 0xFFFFFFFFu;
        }
#pragma unroll
        for (int k = 0; k < GI_B; ++k) TICK(x[k], g[k], o[k]);
#pragma unroll
        for (int k = 0; k < GI_B; ++k)
#pragma unroll
            for (int q = 0; q < GRAPH_NOUT; ++q) __stcs(dst + ((t + k) * GRAPH_NOUT + q) * n, o[k][q]);
    }
    for (; t < p.F; ++t) {
        uint32_t x[GRAPH_NINA], g, o[GRAPH_NOUT];
#pragma unroll
        for (int j = 0; j < GRAPH_NIN; ++j) x[j] = __ldcs(src + (t * GRAPH_NIN + j) * n);
        g = GRAPH_HAS_CHANGED ? __ldcs(chg + t * n) : 0xFFFFFFFFu;
        TICK(x, g, o);
#pragma unroll
        for (int q = 0; q < GRAPH_NOUT; ++q) __stcs(dst + (t * GRAPH_NOUT + q) * n, o[q]);
    }
    GRAPH_STORE_STATE(p.st, p.npad, i)
}

// Four adjacent instances per thread (128-bit accesses): a block covers 2 KiB of every stream row
// instead of 512 B -- fewer distant row segments and pages per block (see pbulk::k_interleaved4).
// n % 4 == 0, 16-byte aligned streams.
#define GI4_B 4
extern "C" __global__ void __launch_bounds__(128) graph_interleaved4(const GraphParams p) {
    const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= p.n) return;
    GState Sa = {}, Sb = {}, Sc = {}, Sd = {};
    GRAPH_LOAD_STATE4(p.st, p.npad, i)
    GParam Pa = {}, Pb = {}, Pc = {}, Pd = {};
    GRAPH_LOAD_PARAM4(p.prm, p.npad, i)
    const uint32_t *src = p.in + i;
    const uint32_t *chg = GRAPH_HAS_CHANGED ? p.changed + i : 0;
    uint32_t *dst = p.out + i;
    const uint64_t n = p.n;
    auto frame = [&](uint64_t t) {
        uint32_t xa[GRAPH_NINA], xb[GRAPH_NINA], xc[GRAPH_NINA], xd[GRAPH_NINA], oa[GRAPH_NOUT], ob[GRAPH_NOUT], oc[GRAPH_NOUT], od[GRAPH_NOUT];
        uint4 g = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
#pragma unroll
        for (int j = 0; j < GRAPH_NIN; ++j) { const uint4 v = __ldcs((const uint4 *)(src + (t * GRAPH_NIN + j) * n)); xa[j] = v.x; xb[j] = v.y; xc[j] = v.z; xd[j] = v.w; }
        if (GRAPH_HAS_CHANGED) g = __ldcs((const uint4 *)(chg + t * n));
        graph_tick(Sa, Pa, xa, g.x, oa); graph_tick(Sb, Pb, xb, g.y, ob); graph_tick(Sc, Pc, xc, g.z, oc); graph_tick(Sd, Pd, xd, g.w, od);
#pragma unroll
        for (int q = 0; q < GRAPH_NOUT; ++q) __stcs((uint4 *)(dst + (t * GRAPH_NOUT + q) * n), make_uint4(oa[q], ob[q], oc[q], od[q]));
    };
    uint64_t t = 0;
    for (; t + GI4_B <= p.F; t += GI4_B) {
        // loads of a batch are independent of the stores of the previous frames only if issued first: keep the
        // batch short (the state of four instances is already in registers) and let the unroller interleave
#pragma unroll
        for (int k = 0; k < GI4_B; ++k) frame(t + k);
    }
    for (; t < p.F; ++t) frame(t);
    GRAPH_STORE_STATE4(p.st, p.npad, i)
}

__device__ __forceinline__ uint32_t smem_u32(const void *q) { return (uint32_t)__cvta_generic_to_shared(q); }
#define TF GRAPH_TF                 // frames per tile: 64, or 32 for graphs with many instructions per tick (more resident warps)
#define ROWS_IN (GRAPH_NIN + (GRAPH_HAS_CHANGED ? 1 : 0))
#define ROWS (ROWS_IN > GRAPH_NOUT ? ROWS_IN : GRAPH_NOUT)   // output q overwrites row q in place
#define STAGES GRAPH_STAGES
#define WARPS GRAPH_WARPS

// [inst][n_inputs][F] in, [inst][F] changed / out (what a host hands over), staged through shared memory with TENSOR TMA
// (planar_bulk.cuh, k_planar_tma): lane r of a warp owns instance r of the warp's 32.  The streams are 3-D tensors
// [inst][stream][F], a box is 32 frames x 1 stream x 32 instances (SWIZZLE_128B), ONE elected lane moves the TF / 32 boxes
// of every stream of a tile, lane r finds 16-byte chunk c of its row at r*128 + ((c ^ (r&7)) << 4); output q
// overwrites the row of stream q in place and leaves with tensor-TMA stores.
struct __align__(64) CUtensorMap { unsigned long long opaque[16]; };
#define TT_BOXB 4096
#define TT_STREAMB ((TF / 32) * TT_BOXB)
#define TT_STAGEB (ROWS * TT_STREAMB)
extern "C" __global__ void __launch_bounds__(WARPS * 32) graph_planar_tma(const GraphParams p, const __grid_constant__ CUtensorMap tm_in,
                                                                           const __grid_constant__ CUtensorMap tm_chg, const __grid_constant__ CUtensorMap tm_out) {
    extern __shared__ __align__(1024) unsigned char sm[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t g0 = ((uint64_t)blockIdx.x * WARPS + warp) * 32;
    if (g0 >= p.n) return;
    const uint32_t rows = p.n - g0 < 32 ? (uint32_t)(p.n - g0) : 32u;
    const bool mine = lane < rows;
    const uint64_t i = g0 + lane;
    const uint32_t sm0 = (smem_u32(sm) + 1023u) & ~1023u;
    const uint32_t base = sm0 + warp * (STAGES * TT_STAGEB);
    const uint32_t bar0 = sm0 + WARPS * STAGES * TT_STAGEB + warp * (STAGES * 8);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0 + 8 * s), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    GRAPH_DECL_STATE
    GParam P = {};
    if (mine) { GRAPH_LOAD_STATE(p.st, p.npad, i) GRAPH_LOAD_PARAM(p.prm, p.npad, i) }
    const uint32_t n_tiles = (uint32_t)((p.F + TF - 1) / TF);
    const unsigned long long tmo = (unsigned long long)&tm_out;
#if GRAPH_ST_HINT
    unsigned long long st_policy;                                     // write-once output: evict-first in L2
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(st_policy));
#endif
    auto cols_of = [&](uint32_t k) { const uint64_t left = p.F - (uint64_t)k * TF; return left < TF ? (uint32_t)left : (uint32_t)TF; };
#if ROWS_IN != 0
    const unsigned long long tmi = (unsigned long long)&tm_in, tmc = (unsigned long long)&tm_chg;
    auto issue = [&](uint32_t k) {                                    // lane 0 only
        const uint32_t s = k % STAGES, nbox = (cols_of(k) + 31) / 32;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8 * s), "r"(ROWS_IN * nbox * TT_BOXB) : "memory");
#pragma unroll
        for (int j = 0; j < ROWS_IN; ++j)
            for (uint32_t h = 0; h < nbox; ++h)
                asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                             ::"r"(base + s * TT_STAGEB + j * TT_STREAMB + h * TT_BOXB), "l"(j < GRAPH_NIN ? tmi : tmc), "r"((int)(k * TF + h * 32)),
                               "r"(j < GRAPH_NIN ? j : 0), "r"((int)g0), "r"(bar0 + 8 * s) : "memory");
    };
    if (lane == 0) for (uint32_t k = 0; k + 2 < STAGES && k < n_tiles; ++k) issue(k);
#endif
#pragma unroll 1
    for (uint32_t k = 0; k < n_tiles; ++k) {
        const uint32_t s = k % STAGES, cols = cols_of(k);
#if ROWS_IN == 0
        // a graph without input streams only stores: every stage is a store buffer, tile k needs the store of tile k-STAGES read out
        if (k >= STAGES) {
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(STAGES - 1) : "memory");
            __syncwarp();
        }
#else
        if (k + STAGES - 2 < n_tiles && lane == 0) {                  // that stage last held tile k-2: its stores must have read it out
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            issue(k + STAGES - 2);
        }
        asm volatile("{\n\t.reg .pred q;\n\tW: mbarrier.try_wait.parity.shared::cta.b64 q, [%0], %1;\n\t@q bra D;\n\tbra W;\n\tD:\n\t}"
                     ::"r"(bar0 + 8 * s), "r"((k / STAGES) & 1) : "memory");
#endif
        const uint32_t row = base + s * TT_STAGEB + lane * 128;       // stream j, chunk c: row + j * TT_STREAMB + (c >> 3) * TT_BOXB + (((c & 7) ^ (lane & 7)) << 4)
        if (mine) {
            for (uint32_t c = 0; c < cols / 4; ++c) {
                const uint32_t at = row + (c >> 3) * TT_BOXB + (((c & 7) ^ (lane & 7)) << 4);
                uint32_t xa[GRAPH_NINA], xb[GRAPH_NINA], xc[GRAPH_NINA], xd[GRAPH_NINA], ga = 0xFFFFFFFFu, gb = 0xFFFFFFFFu, gc = 0xFFFFFFFFu, gd = 0xFFFFFFFFu;
                uint32_t oa[GRAPH_NOUT], ob[GRAPH_NOUT], oc[GRAPH_NOUT], od[GRAPH_NOUT];
#pragma unroll
                for (int j = 0; j < GRAPH_NIN; ++j)
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(xa[j]), "=r"(xb[j]), "=r"(xc[j]), "=r"(xd[j]) : "r"(at + j * TT_STREAMB));
                if (GRAPH_HAS_CHANGED)
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(ga), "=r"(gb), "=r"(gc), "=r"(gd) : "r"(at + GRAPH_NIN * TT_STREAMB));
                TICK(xa, ga, oa); TICK(xb, gb, ob); TICK(xc, gc, oc); TICK(xd, gd, od);
#pragma unroll
                for (int q = 0; q < GRAPH_NOUT; ++q)
                    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(at + q * TT_STREAMB), "r"(oa[q]), "r"(ob[q]), "r"(oc[q]), "r"(od[q]) : "memory");
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            const uint32_t nbox = (cols + 31) / 32;
#pragma unroll
            for (int q = 0; q < GRAPH_NOUT; ++q)
                for (uint32_t h = 0; h < nbox; ++h) {
#if GRAPH_ST_HINT
                    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%1, %2, %3}], [%4], %5;"
                                 ::"l"(tmo), "r"((int)(k * TF + h * 32)), "r"(q), "r"((int)g0), "r"(base + s * TT_STAGEB + q * TT_STREAMB + h * TT_BOXB), "l"(st_policy) : "memory");
#else
                    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];"
                                 ::"l"(tmo), "r"((int)(k * TF + h * 32)), "r"(q), "r"((int)g0), "r"(base + s * TT_STAGEB + q * TT_STREAMB + h * TT_BOXB) : "memory");
#endif
                }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    if (mine) { GRAPH_STORE_STATE(p.st, p.npad, i) }
}

// planar streams of any length / alignment: one thread per instance, scalar accesses
extern "C" __global__ void __launch_bounds__(128) graph_planar_simple(const GraphParams p) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    GRAPH_DECL_STATE
    GRAPH_LOAD_STATE(p.st, p.npad, i)
    GParam P = {};
    GRAPH_LOAD_PARAM(p.prm, p.npad, i)
    for (uint64_t t = 0; t < p.F; ++t) {
        uint32_t x[GRAPH_NINA], g, o[GRAPH_NOUT];
#pragma unroll
        for (int j = 0; j < GRAPH_NIN; ++j) x[j] = p.in[(i * GRAPH_NIN + j) * p.F + t];
        g = GRAPH_HAS_CHANGED ? p.changed[i * p.F + t] : 0xFFFFFFFFu;
        TICK(x, g, o);
#pragma unroll
        for (int q = 0; q < GRAPH_NOUT; ++q) p.out[(i * GRAPH_NOUT + q) * p.F + t] = o[q];
    }
    GRAPH_STORE_STATE(p.st, p.npad, i)
}

// Bus mix (io.mix; GraphMixParams as in k_graph.cu): one thread per instance for frames [m.t0, m.t0 + m.fc), MIX_CF frames
// at a time, the per-instance outputs never leave registers.  The bus tree's first five levels run across the warp's lanes
// as a recursive-halving transpose-reduce, lane bit 0 first (level 1 adds lanes 2m, 2m+1): at level b a lane keeps the half
// of its frames that its lane bit b selects and adds the partner's sums for them -- one shuffle and one add per output per
// instance-frame -- until every lane holds one frame, then butterflies for the lane bits left.  Lane r ends with frame
// sum_b bit_b(r) * (MIX_CF >> (b + 1)).  The block's warps then add up in shared memory in groups of m.wg warps (the next
// levels), and the group sums go to m.dst; k_graph_mix_tree does the levels above.  Lanes past n add the tree's padding,
// -0.0f for a float and 0 for a w output, an exact identity.
struct GraphMixParams { uint32_t *dst; uint64_t t0, fc, dst_F, dst_t0; uint32_t wg, outf; };   // must match k_graph.cu
#define MIX_CF (GRAPH_NOUT <= 2 ? 16 : GRAPH_NOUT <= 4 ? 8 : 4)   // frames per transpose: MIX_CF * GRAPH_NOUT sums in registers
#define MIX_WARPS 4
#define MIX_F(q) ((GRAPH_OUTF >> (q)) & 1u)
__device__ __forceinline__ uint32_t mix_add(uint32_t a, uint32_t b, bool f) {
    return f ? __float_as_uint(__fadd_rn(__uint_as_float(a), __uint_as_float(b))) : a + b;
}
extern "C" __global__ void __launch_bounds__(MIX_WARPS * 32) graph_mix(const GraphParams p, const GraphMixParams m) {
    __shared__ uint32_t red[2][MIX_WARPS][GRAPH_NOUT][MIX_CF];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool mine = i < p.n;
    GRAPH_DECL_STATE
    GParam P = {};
    if (mine) { GRAPH_LOAD_STATE(p.st, p.npad, i) GRAPH_LOAD_PARAM(p.prm, p.npad, i) }
    const bool il = p.layout == 1;
    const uint64_t n = p.n, t1 = m.t0 + m.fc;
    uint32_t f_lane = 0;
#pragma unroll
    for (int b = 0, h = MIX_CF / 2; h >= 1; ++b, h >>= 1) f_lane += ((lane >> b) & 1u) * h;
    // slices start at m.t0 + a multiple of MIX_CF, and m.t0 is 0 or a multiple of 32 (k_graph.cu)
    const bool vec4 = ROWS_IN != 0 && !il && p.F % 4 == 0 && m.t0 % 4 == 0 && ((unsigned long long)p.in & 15) == 0 && ((unsigned long long)p.changed & 15) == 0;
#pragma unroll 1
    for (uint64_t tc = m.t0, c = 0; tc < t1; tc += MIX_CF, ++c) {
        uint32_t v[GRAPH_NOUT][MIX_CF];
        // the slice's input words are loaded before any tick, so their latencies overlap
        uint32_t x[MIX_CF][GRAPH_NINA], g[MIX_CF];
        if (vec4 && mine && tc + MIX_CF <= t1) {                         // PLANAR rows, 16-byte aligned: four frames per load
#pragma unroll
            for (int c = 0; c < MIX_CF / 4; ++c) {
#pragma unroll
                for (int j = 0; j < GRAPH_NIN; ++j) {
                    const uint4 w = *(const uint4 *)(p.in + (i * GRAPH_NIN + j) * p.F + tc + 4 * c);
                    x[4 * c][j] = w.x; x[4 * c + 1][j] = w.y; x[4 * c + 2][j] = w.z; x[4 * c + 3][j] = w.w;
                }
                uint4 w = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
                if (GRAPH_HAS_CHANGED) w = *(const uint4 *)(p.changed + i * p.F + tc + 4 * c);
                g[4 * c] = w.x; g[4 * c + 1] = w.y; g[4 * c + 2] = w.z; g[4 * c + 3] = w.w;
            }
        } else
#pragma unroll
        for (int k = 0; k < MIX_CF; ++k) {
            const uint64_t t = tc + k;
            const bool live = mine && t < t1;
#pragma unroll
            for (int j = 0; j < GRAPH_NIN; ++j) x[k][j] = !live ? 0u : il ? __ldcs(p.in + (t * GRAPH_NIN + j) * n + i) : p.in[(i * GRAPH_NIN + j) * p.F + t];
            g[k] = GRAPH_HAS_CHANGED && live ? (il ? __ldcs(p.changed + t * n + i) : p.changed[i * p.F + t]) : 0xFFFFFFFFu;
        }
#pragma unroll
        for (int k = 0; k < MIX_CF; ++k) {
            const uint64_t t = tc + k;
            uint32_t o[GRAPH_NOUT];
            if (mine && t < t1) {
                TICK(x[k], g[k], o);
                if (p.out) {
#pragma unroll
                    for (int q = 0; q < GRAPH_NOUT; ++q) p.out[il ? (t * GRAPH_NOUT + q) * n + i : (i * GRAPH_NOUT + q) * p.F + t] = o[q];
                }
            } else {
#pragma unroll
                for (int q = 0; q < GRAPH_NOUT; ++q) o[q] = MIX_F(q) ? 0x80000000u : 0u;
            }
#pragma unroll
            for (int q = 0; q < GRAPH_NOUT; ++q) v[q][k] = o[q];
        }
#pragma unroll
        for (int b = 0, h = MIX_CF / 2; h >= 1; ++b, h >>= 1) {
            const bool hi = (lane >> b) & 1u;
#pragma unroll
            for (int k = 0; k < h; ++k)
#pragma unroll
                for (int q = 0; q < GRAPH_NOUT; ++q) {
                    const uint32_t send = hi ? v[q][k] : v[q][k + h], keep = hi ? v[q][k + h] : v[q][k];
                    v[q][k] = mix_add(keep, __shfl_xor_sync(0xFFFFFFFFu, send, 1 << b), MIX_F(q));
                }
        }
#pragma unroll
        for (int b = 32 / MIX_CF; b > 1; b >>= 1)                       // lane bits above log2(MIX_CF)
#pragma unroll
            for (int q = 0; q < GRAPH_NOUT; ++q) v[q][0] = mix_add(v[q][0], __shfl_xor_sync(0xFFFFFFFFu, v[q][0], 32 / b), MIX_F(q));
        if (lane < MIX_CF)
#pragma unroll
            for (int q = 0; q < GRAPH_NOUT; ++q) red[c & 1][warp][q][f_lane] = v[q][0];
        __syncthreads();                                                 // red[c & 1] was last read in slice c - 2, before slice c - 1's barrier
        const uint32_t per_block = MIX_WARPS >> (__ffs(m.wg) - 1);        // m.wg is a power of two
        for (uint32_t e = threadIdx.x; e < per_block * GRAPH_NOUT * MIX_CF; e += blockDim.x) {
            const uint32_t f = e % MIX_CF, q = (e / MIX_CF) % GRAPH_NOUT, gq = e / (MIX_CF * GRAPH_NOUT);
            const bool isf = MIX_F(q);
            uint32_t w[MIX_WARPS];
#pragma unroll
            for (int k = 0; k < MIX_WARPS; ++k) w[k] = k < (int)m.wg ? red[c & 1][gq * m.wg + k][q][f] : (isf ? 0x80000000u : 0u);
#pragma unroll
            for (int h = MIX_WARPS / 2; h >= 1; h >>= 1)
#pragma unroll
                for (int k = 0; k < h; ++k) w[k] = mix_add(w[2 * k], w[2 * k + 1], isf);
            const uint64_t grp = (uint64_t)blockIdx.x * per_block + gq;
            if (grp * 32 * m.wg < n && tc + f < t1) m.dst[(grp * GRAPH_NOUT + q) * m.dst_F + m.dst_t0 + (tc - m.t0) + f] = w[0];
        }
    }
    if (mine) { GRAPH_STORE_STATE(p.st, p.npad, i) }
}

extern "C" __global__ void graph_planar_smem(uint32_t *out) { out[0] = WARPS * 32; out[1] = WARPS * STAGES * TT_STAGEB + WARPS * STAGES * 8 + 1024; out[2] = MIX_WARPS; }
)SRC";

}  // namespace

// Source for one graph: state words s0..s{W-1} in node order (acc {out}; edge {out, last}; ...), param words p0..p{Q-1}.
std::string cproc_graph_jit_source(const std::vector<cproc_cuda_node> &nodes, uint32_t n_inputs, const std::vector<uint32_t> &outs, bool has_changed) {
    std::vector<uint32_t> off(nodes.size()), poff(nodes.size());
    uint32_t words = 0, pwords = 0;
    for (size_t k = 0; k < nodes.size(); ++k) { off[k] = words; words += cproc_node_words(nodes[k].type); poff[k] = pwords; pwords += cproc_node_param_words(nodes[k].type); }
    char buf[1024];
    // state words live in a struct so that a kernel can keep several instances per thread
    std::string decl = "struct GState { uint32_t", load = "#define GRAPH_LOAD_STATE(st, npad, i)", store = "#define GRAPH_STORE_STATE(st, npad, i)";
    std::string load4 = "#define GRAPH_LOAD_STATE4(st, npad, i) { uint4 v;", store4 = "#define GRAPH_STORE_STATE4(st, npad, i) {";
    for (uint32_t w = 0; w < words; ++w) {
        snprintf(buf, sizeof(buf), "%s s%u", w ? "," : "", w); decl += buf;
        snprintf(buf, sizeof(buf), " S.s%u = (st)[%uull * (npad) + (i)];", w, w); load += buf;
        snprintf(buf, sizeof(buf), " (st)[%uull * (npad) + (i)] = S.s%u;", w, w); store += buf;
        snprintf(buf, sizeof(buf), " v = *(const uint4 *)((st) + %uull * (npad) + (i)); Sa.s%u = v.x; Sb.s%u = v.y; Sc.s%u = v.z; Sd.s%u = v.w;", w, w, w, w, w); load4 += buf;
        snprintf(buf, sizeof(buf), " *(uint4 *)((st) + %uull * (npad) + (i)) = make_uint4(Sa.s%u, Sb.s%u, Sc.s%u, Sd.s%u);", w, w, w, w, w); store4 += buf;
    }
    decl += "; };\n#define GRAPH_DECL_STATE GState S = {};\n"; load += "\n"; store += "\n"; load4 += " }\n"; store4 += " }\n";
    // param words (constant over a launch): one register each
    std::string pdecl = "struct GParam { uint32_t", pload = "#define GRAPH_LOAD_PARAM(prm, npad, i)", pload4 = "#define GRAPH_LOAD_PARAM4(prm, npad, i) { uint4 v;";
    if (pwords == 0) pdecl += " none";
    for (uint32_t w = 0; w < pwords; ++w) {
        snprintf(buf, sizeof(buf), "%s p%u", w ? "," : "", w); pdecl += buf;
        snprintf(buf, sizeof(buf), " P.p%u = (prm)[%uull * (npad) + (i)];", w, w); pload += buf;
        snprintf(buf, sizeof(buf), " v = *(const uint4 *)((prm) + %uull * (npad) + (i)); Pa.p%u = v.x; Pb.p%u = v.y; Pc.p%u = v.z; Pd.p%u = v.w;", w, w, w, w, w); pload4 += buf;
    }
    pdecl += "; };\n"; pload += "\n"; pload4 += " }\n";
    if (pwords == 0) pload4 = "#define GRAPH_LOAD_PARAM4(prm, npad, i)\n";
    std::string tick = "#define GRAPH_TICK(x, g)";
    for (size_t k = 0; k < nodes.size(); ++k) {
        const cproc_cuda_node &nd = nodes[k];
        const uint32_t kind = CPROC_CUDA_NODE_KIND(nd.type);
        // an operand as a `w` (want_f = false) or as a float (true); w -> float converts by value like the C initialiser does
        auto operand = [&](int32_t src, bool want_f) {
            char ob[96];
            if (src == CPROC_CUDA_SRC_ZERO) return std::string(want_f ? "0.0f" : "0u");
            const bool src_f = src >= 0 && cproc_kind_out_float(nodes[src].type);
            char raw[64];
            if (src >= 0) snprintf(raw, sizeof(raw), "s%u", off[src]);
            else snprintf(raw, sizeof(raw), "(x)[%d]", -(src + 1));
            if (!want_f) return std::string(raw);
            snprintf(ob, sizeof(ob), src_f ? "__uint_as_float(%s)" : "__uint2float_rn(%s)", raw);
            return std::string(ob);
        };
        const std::string in = operand(nd.src, kind < CPROC_CUDA_NODE_KINDS && (k_cproc_kinds[kind].input_f & 1u));
        std::string cond;
        if (nd.cond_mask == 0xFFFFFFFFu && !has_changed) cond = "";
        else { snprintf(buf, sizeof(buf), "if ((g) & 0x%xu) ", nd.cond_mask); cond = buf; }
        const uint32_t o = off[k], q = poff[k];
        if (kind == CPROC_CUDA_NODE_PDM) {
            // pdm.h:13-77: q = sK >> sh; a = (q << sh) + dither; s1 += in - a; sk += s(k-1) - a; out = q
            const uint32_t K = CPROC_CUDA_NODE_ARG(nd.type) & 7u, sh = CPROC_CUDA_NODE_ARG(nd.type) >> 3;
            std::string body;
            snprintf(buf, sizeof(buf), " %s{ const uint32_t vin = %s; const uint32_t q = s%u >> %u; const uint32_t a = (q << %u)", cond.c_str(), in.c_str(), o + K, sh, sh);
            body = buf;
            if (K > 1) body += " + " + operand(nd.src2, false);
            snprintf(buf, sizeof(buf), "; s%u += vin - a;", o + 1);
            body += buf;
            for (uint32_t kk = 2; kk <= K; ++kk) { snprintf(buf, sizeof(buf), " s%u += s%u - a;", o + kk, o + kk - 1); body += buf; }
            snprintf(buf, sizeof(buf), " s%u = q; }", o);
            body += buf;
            tick += body;
            continue;
        }
        switch (kind) {
        case CPROC_CUDA_NODE_GLIDE: {
            const uint32_t L = CPROC_CUDA_NODE_ARG(nd.type);                  // mod_pdm_pwm.c:129-143, mod_controlrate.c:28-40
            snprintf(buf, sizeof(buf), " %s{ if (s%u == 0) { s%u = s%u; s%u = s%u; s%u += s%u << %u; s%u = (uint32_t)((int32_t)(%s - s%u) >> %u); } s%u += s%u; s%u = (s%u + 1) & 0x%xu; }",
                     cond.c_str(), o + 4, o, o + 2, o + 1, o + 3, o + 2, o + 3, L, o + 3, in.c_str(), o + 2, L, o, o + 1, o + 4, o + 4, (1u << L) - 1u);
            break; }
        case CPROC_CUDA_NODE_EDGE: snprintf(buf, sizeof(buf), " %s{ const uint32_t v = %s; s%u = (v != s%u); s%u = v; }", cond.c_str(), in.c_str(), o, o + 1, o + 1); break;   // cproc.h:151-154
        // extension processors, include/cproc_ext.h: one IEEE rounding per statement
        case CPROC_CUDA_NODE_PHASOR_F:
            snprintf(buf, sizeof(buf), " %s{ s%u = __float_as_uint(__fmul_rn(__int2float_rn((int32_t)s%u), 4.656612873077392578125e-10f)); s%u += P.p%u + %s; }", cond.c_str(), o, o + 1, o + 1, q, in.c_str());
            break;
        case CPROC_CUDA_NODE_SVF:
            snprintf(buf, sizeof(buf), " %s{ const float vf = __uint_as_float(P.p%u), vq = __uint_as_float(P.p%u), vbp = __uint_as_float(s%u); const float lp = __fmaf_rn(vf, vbp, __uint_as_float(s%u));"
                     " float hp = __fsub_rn(%s, lp); hp = __fmaf_rn(-vq, vbp, hp); s%u = __float_as_uint(__fmaf_rn(vf, hp, vbp)); s%u = __float_as_uint(lp); }",
                     cond.c_str(), q, q + 1, o + 1, o, in.c_str(), o + 1, o);
            break;
        case CPROC_CUDA_NODE_ENV:
            snprintf(buf, sizeof(buf), " %s{ float e = __uint_as_float(s%u); if (s%u < P.p%u) { e = __fadd_rn(e, __uint_as_float(P.p%u)); if (e > 1.0f) e = 1.0f; }"
                     " else { e = __fsub_rn(e, __uint_as_float(P.p%u)); if (e < 0.0f) e = 0.0f; } s%u = __float_as_uint(e); s%u += 1u; s%u = __float_as_uint(__fmul_rn(%s, e)); }",
                     cond.c_str(), o + 1, o + 2, q + 2, q, q + 1, o + 1, o + 2, o, in.c_str());
            break;
        case CPROC_CUDA_NODE_ONEPOLE:
            snprintf(buf, sizeof(buf), " %s{ const float y = __uint_as_float(s%u); s%u = __float_as_uint(__fmaf_rn(__uint_as_float(P.p%u), __fsub_rn(%s, y), y)); }", cond.c_str(), o, o, q, in.c_str());
            break;
        case CPROC_CUDA_NODE_GAIN:
            snprintf(buf, sizeof(buf), " %s{ s%u = __float_as_uint(__fmul_rn(__uint_as_float(P.p%u), %s)); }", cond.c_str(), o, q, in.c_str());
            break;
        case CPROC_CUDA_NODE_ASFLOAT:
            snprintf(buf, sizeof(buf), " %s{ s%u = %s; }", cond.c_str(), o, in.c_str());
            break;
        case CPROC_CUDA_NODE_GLIDE_F: {
            const uint32_t L = CPROC_CUDA_NODE_ARG(nd.type);
            snprintf(buf, sizeof(buf), " %s{ if (s%u == 0) s%u = __float_as_uint(__fmul_rn(__fsub_rn(%s, __uint_as_float(s%u)), %.9ef)); s%u = __float_as_uint(__fadd_rn(__uint_as_float(s%u), __uint_as_float(s%u)));"
                     " s%u = (s%u + 1) & 0x%xu; }", cond.c_str(), o + 2, o + 1, in.c_str(), o, 1.0 / (double)(1u << L), o, o, o + 1, o + 2, o + 2, (1u << L) - 1u);
            break; }
        case CPROC_CUDA_NODE_MUL:
            snprintf(buf, sizeof(buf), " %s{ s%u = __float_as_uint(__fmul_rn(%s, %s)); }", cond.c_str(), o, in.c_str(), operand(nd.src2, true).c_str());
            break;
        default: snprintf(buf, sizeof(buf), " %s{ s%u += %s; }", cond.c_str(), o, in.c_str()); break;                                                                            // cproc.h:140-142
        }
        tick += buf;
    }
    tick += "\n";
    std::string outm = "#define GRAPH_OUTS(o)";
    for (size_t q = 0; q < outs.size(); ++q) { snprintf(buf, sizeof(buf), " (o)[%zu] = s%u;", q, off[outs[q]]); outm += buf; }
    // Block shape of the PLANAR staging kernels.  A tick of a float voice is ~20 dependent instructions and its graph has no input
    // stream: measured on the C4 voice graph (tools/sweep_graph_tiles.sh, profiles/r2_sweep_graph_tiles.txt) one warp per block with
    // 64-frame tiles and three stages is the best shape (5.74 TB/s with every stage a store buffer -- a store-only graph waits for the
    // store of tile k-3, not k-2; two stages x two warps 5.68, 32-frame tiles 4.9-5.4, profiles/r2_sweep_graph_tiles.txt).
    static const uint8_t k_cost[CPROC_CUDA_NODE_KINDS] = {1, 2, 6, 7, 3, 5, 6, 2, 1, 0, 4, 1};
    uint32_t cost = 0;
    for (const cproc_cuda_node &nd : nodes) cost += k_cost[CPROC_CUDA_NODE_KIND(nd.type)];
    int tf = 64, stages = 3, warps = cost >= 12 ? 1 : 2;
    // experiments: CPROC_GRAPH_TF / _STAGES / _WARPS override the tile shape of the generated PLANAR kernels
    if (const char *e = getenv("CPROC_GRAPH_TF")) { const int v = atoi(e); if (v == 32 || v == 64 || v == 128) tf = v; }
    if (const char *e = getenv("CPROC_GRAPH_STAGES")) { const int v = atoi(e); if (v >= 2 && v <= 6) stages = v; }
    if (const char *e = getenv("CPROC_GRAPH_WARPS")) { const int v = atoi(e); if (v >= 1 && v <= 8) warps = v; }
    int hint = 0;
    if (const char *e = getenv("CPROC_GRAPH_ST_HINT")) hint = atoi(e) != 0;
    uint32_t outf = 0;                                     // output q is a float: the node kind's out is (as in operand())
    for (size_t q = 0; q < outs.size(); ++q) if (cproc_kind_out_float(nodes[outs[q]].type)) outf |= 1u << q;
    snprintf(buf, sizeof(buf), "\n#define GRAPH_NOUT %zu\n#define GRAPH_NIN %u\n#define GRAPH_NINA %u\n#define GRAPH_HAS_CHANGED %d\n#define GRAPH_TF %d\n#define GRAPH_STAGES %d\n#define GRAPH_WARPS %d\n#define GRAPH_ST_HINT %d\n#define GRAPH_OUTF 0x%xu\n",
             outs.size(), n_inputs, n_inputs ? n_inputs : 1u, has_changed ? 1 : 0, tf, stages, warps, hint, outf);
    // the tick text names the state words s<k>: they are members of the GState `S` in scope
    static const std::regex word("\\bs([0-9]+)\\b");
    tick = std::regex_replace(tick, word, "S.s$1");
    outm = std::regex_replace(outm, word, "S.s$1");
    return k_jit_head + decl + load + store + load4 + store4 + pdecl + pload + pload4 + tick + outm + buf + k_jit_tail;
}

// Compile (once per batch and `changed` presence) and return the two kernels.
int cproc_graph_jit_get(cproc_cuda_batch *b, bool has_changed, cproc_graph_jit **out) {
    cproc_cuda_ctx *ctx = b->ctx;
    cproc_graph_jit &j = b->jit[has_changed ? 1 : 0];
    if (j.state == 2) return -1;                           // failed before: stay on the table kernel
    if (j.state == 0) {
        j.state = 2;
        if (!nvrtc_load()) { b->jit_log = "libnvrtc not found"; return -1; }
        const std::string src = cproc_graph_jit_source(b->nodes, b->cfg.n_inputs, b->outs, has_changed);
        // cubins are cached per process by their source text: a patcher that grows a graph node by
        // node, or many batches of the same graph, compile once
        static std::unordered_map<std::string, std::vector<char>> cubin_cache;
        auto hit = cubin_cache.find(src);
        if (hit != cubin_cache.end()) j.cubin = hit->second;
        void *prog = nullptr;
        if (j.cubin.empty()) {
        if (g_nvrtc.create(&prog, src.c_str(), "cproc_graph.cu", 0, nullptr, nullptr)) { b->jit_log = "nvrtcCreateProgram failed"; return -1; }
        const char *opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "-default-device"};
        const int rc = g_nvrtc.compile(prog, 4, opts);
        size_t ls = 0;
        g_nvrtc.log_size(prog, &ls);
        if (ls > 1) { b->jit_log.resize(ls); g_nvrtc.log(prog, &b->jit_log[0]); }
        if (rc) { g_nvrtc.destroy(&prog); return -1; }
        size_t cs = 0;
        g_nvrtc.cubin_size(prog, &cs);
        j.cubin.resize(cs);
        g_nvrtc.cubin(prog, j.cubin.data());
        g_nvrtc.destroy(&prog);
        cubin_cache[src] = j.cubin;
        }
        if (cudaLibraryLoadData(&j.lib, j.cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0) != cudaSuccess) { cudaGetLastError(); b->jit_log = "cudaLibraryLoadData failed"; return -1; }
        cudaKernel_t kq = nullptr;
        if (cudaLibraryGetKernel(&j.k_il, j.lib, "graph_interleaved") != cudaSuccess ||
            cudaLibraryGetKernel(&j.k_ps, j.lib, "graph_planar_simple") != cudaSuccess || cudaLibraryGetKernel(&j.k_pt, j.lib, "graph_planar_tma") != cudaSuccess ||
            cudaLibraryGetKernel(&j.k_il4, j.lib, "graph_interleaved4") != cudaSuccess || cudaLibraryGetKernel(&j.k_mix, j.lib, "graph_mix") != cudaSuccess ||
            cudaLibraryGetKernel(&kq, j.lib, "graph_planar_smem") != cudaSuccess) { cudaGetLastError(); b->jit_log = "cudaLibraryGetKernel failed"; return -1; }
        // block and shared-memory size of graph_planar_tma and the mix kernel's block are defined by the generated source: ask it
        uint32_t *d = nullptr, h[3] = {0, 0, 0};
        if (cudaMalloc(&d, sizeof(h)) != cudaSuccess) { cudaGetLastError(); return -1; }
        void *args[] = {&d};
        cudaError_t e = cudaLaunchKernel((const void *)kq, dim3(1), dim3(1), args, 0, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        cudaFree(d);
        if (e != cudaSuccess) { cudaGetLastError(); b->jit_log = "graph_planar_smem query failed"; return -1; }
        j.pt_block = h[0]; j.pt_smem = h[1]; j.mix_warps = h[2];
        if (j.pt_smem > 227 * 1024) { b->jit_log = "planar staging does not fit shared memory (too many input streams)"; j.k_pt = nullptr; }
        else if (cudaFuncSetAttribute((const void *)j.k_pt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)j.pt_smem) != cudaSuccess) { cudaGetLastError(); j.k_pt = nullptr; }
        j.state = 1;
    }
    *out = &j;
    return 0;
}

extern "C" const char *cproc_cuda_graph_jit_log(const cproc_cuda_batch *b) { return b ? b->jit_log.c_str() : ""; }
extern "C" int cproc_cuda_graph_jit_source(const cproc_cuda_node *nodes, uint32_t n_nodes, uint32_t n_inputs, const uint32_t *out_nodes,
                                           uint32_t n_outputs, int has_changed, char *dst, size_t cap) {
    if (!nodes || n_nodes == 0 || n_nodes > CPROC_CUDA_GRAPH_MAX_NODES || !out_nodes || n_outputs == 0 || n_outputs > CPROC_CUDA_GRAPH_MAX_OUTPUTS)
        return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_jit_source: bad node table");
    for (uint32_t q = 0; q < n_outputs; ++q) if (out_nodes[q] >= n_nodes) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_jit_source: output node %u of %u", out_nodes[q], n_nodes);
    for (uint32_t k = 0; k < n_nodes; ++k)
        if (const char *why = cproc_node_check(nodes, k, n_inputs))
            return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "graph_jit_source: node %u: %s", k, why);
    const std::string s = cproc_graph_jit_source(std::vector<cproc_cuda_node>(nodes, nodes + n_nodes), n_inputs, std::vector<uint32_t>(out_nodes, out_nodes + n_outputs), has_changed != 0);
    if (dst && cap) { const size_t n = s.size() < cap - 1 ? s.size() : cap - 1; memcpy(dst, s.data(), n); dst[n] = 0; }
    return (int)s.size();
}
