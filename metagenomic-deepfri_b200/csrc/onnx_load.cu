// mdf_model_load / mdf_cnn_model_load / mdf_onnx_inspect: the `.onnx` file behind the C ABI.
//
// The reference hands `<model>.onnx` to onnxruntime (mDeepFRI/predict.pyx:62-73).  Here the file is decoded from the protobuf
// wire format (public onnx.proto, IR 8; no protobuf library), the graph is *recognised* as a DeepFRI GCN head (LSTM-LM ->
// embedding -> GraphConv stack -> sum-pool -> dense -> FuncPredictor, SURVEY.md §3.3) or a sequence-only DeepCNN head, and the
// weights are handed to mdf_model_create / mdf_cnn_model_create.  Every weight is located by its role in the dataflow (what it is
// connected to and its shape), never by name; every hyper-parameter is read from initialisers / op types.  The adjacency
// normalisation sub-graph is not assumed: it is evaluated (host, float64, a 6- and a 9-residue probe map) and must equal
// D (A - diag(A) + I) D with d = 1 / (eps + sqrt(rowsum)) - so any lowering of GraphConv._normalize is accepted and anything
// else (e.g. A + I without the diagonal removal, a column sum) is rejected.  There is no fallback executor: a graph that does
// not fit fails with MDF_EUNSUPPORTED and the reason.
#include <errno.h>
#include <math.h>
#include <stdarg.h>
#include <functional>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "gcn.cuh"

namespace mdf {
namespace onnx {

// ------------------------------------------------------------------------------------------- wire format
struct Reader {
    const uint8_t *p, *end;
    bool ok = true;
    Reader(const uint8_t *b, size_t n) : p(b), end(b + n) {}
    bool more() const { return ok && p < end; }
    uint64_t varint()
    {
        uint64_t r = 0;
        for (int shift = 0; shift < 70; shift += 7) {
            if (p >= end) { ok = false; return 0; }
            const uint8_t b = *p++;
            r |= (uint64_t)(b & 0x7F) << shift;
            if (!(b & 0x80)) return r;
        }
        ok = false;
        return 0;
    }
    // one field: number, wire type and either the scalar value or the [ptr, len) payload
    bool field(int &fno, int &wt, uint64_t &val, const uint8_t *&ptr, size_t &len)
    {
        const uint64_t key = varint();
        if (!ok) return false;
        fno = (int)(key >> 3);
        wt = (int)(key & 7);
        ptr = nullptr; len = 0; val = 0;
        if (wt == 0) { val = varint(); }
        else if (wt == 1) { if (end - p < 8) { ok = false; return false; } memcpy(&val, p, 8); ptr = p; len = 8; p += 8; }
        else if (wt == 2) {
            const uint64_t n = varint();
            if (!ok || (uint64_t)(end - p) < n) { ok = false; return false; }
            ptr = p; len = (size_t)n; p += n;
        } else if (wt == 5) { if (end - p < 4) { ok = false; return false; } uint32_t v; memcpy(&v, p, 4); val = v; ptr = p; len = 4; p += 4; }
        else { ok = false; }
        return ok;
    }
};

enum { DT_FLOAT = 1, DT_UINT8 = 2, DT_INT8 = 3, DT_INT32 = 6, DT_INT64 = 7, DT_BOOL = 9, DT_FLOAT16 = 10, DT_DOUBLE = 11 };

struct Tensor {
    std::string name;
    int dtype = DT_FLOAT;
    std::vector<int64_t> dims;
    bool has_raw = false;
    std::string raw;
    std::vector<float> fdata;
    std::vector<double> ddata;
    std::vector<int64_t> idata;
    int64_t numel() const { int64_t n = 1; for (auto d : dims) n *= d; return n; }
    bool is_float() const { return dtype == DT_FLOAT || dtype == DT_DOUBLE || dtype == DT_FLOAT16; }
    bool to_f64(std::vector<double> &out) const;
    bool to_f32(std::vector<float> &out) const
    {
        std::vector<double> d;
        if (dtype == DT_FLOAT && has_raw) {                    // the common case: no detour through double
            if ((int64_t)raw.size() != numel() * 4) return false;
            out.resize((size_t)numel());
            memcpy(out.data(), raw.data(), raw.size());
            return true;
        }
        if (!to_f64(d)) return false;
        out.assign(d.begin(), d.end());
        return true;
    }
};

static float half_to_float(uint16_t h)
{
    const uint32_t s = (h >> 15) & 1, e = (h >> 10) & 31, m = h & 1023;
    float v;
    if (e == 0) v = ldexpf((float)m, -24);
    else if (e == 31) v = m ? NAN : INFINITY;
    else v = ldexpf((float)(m | 1024), (int)e - 25);
    return s ? -v : v;
}

bool Tensor::to_f64(std::vector<double> &out) const
{
    const int64_t n = numel();
    out.resize((size_t)n);
    auto raw_as = [&](auto tag) {
        using T = decltype(tag);
        if ((int64_t)raw.size() != n * (int64_t)sizeof(T)) return false;
        for (int64_t i = 0; i < n; ++i) { T v; memcpy(&v, raw.data() + i * sizeof(T), sizeof(T)); out[(size_t)i] = (double)v; }
        return true;
    };
    if (has_raw) {
        switch (dtype) {
        case DT_FLOAT: return raw_as(float());
        case DT_DOUBLE: return raw_as(double());
        case DT_INT32: return raw_as(int32_t());
        case DT_INT64: return raw_as(int64_t());
        case DT_UINT8: case DT_BOOL: return raw_as(uint8_t());
        case DT_INT8: return raw_as(int8_t());
        case DT_FLOAT16:
            if ((int64_t)raw.size() != n * 2) return false;
            for (int64_t i = 0; i < n; ++i) { uint16_t h; memcpy(&h, raw.data() + i * 2, 2); out[(size_t)i] = half_to_float(h); }
            return true;
        default: return false;
        }
    }
    if (dtype == DT_FLOAT) { if ((int64_t)fdata.size() != n) return false; for (int64_t i = 0; i < n; ++i) out[(size_t)i] = fdata[(size_t)i]; return true; }
    if (dtype == DT_DOUBLE) { if ((int64_t)ddata.size() != n) return false; out = ddata; return true; }
    if (dtype == DT_FLOAT16) { if ((int64_t)idata.size() != n) return false; for (int64_t i = 0; i < n; ++i) out[(size_t)i] = half_to_float((uint16_t)idata[(size_t)i]); return true; }
    if ((int64_t)idata.size() != n) return false;
    for (int64_t i = 0; i < n; ++i) out[(size_t)i] = (double)idata[(size_t)i];
    return true;
}

struct Attr {
    int type = 0;
    bool has_f = false, has_i = false, has_s = false, has_t = false;
    float f = 0.f;
    int64_t i = 0;
    std::string s;
    Tensor t;
    std::vector<float> floats;
    std::vector<int64_t> ints;
    std::vector<std::string> strings;
};

struct Node {
    std::string op, name;
    std::vector<std::string> in, out;
    std::map<std::string, Attr> attrs;
    int64_t attr_i(const char *k, int64_t dflt) const { auto it = attrs.find(k); return it == attrs.end() ? dflt : it->second.i; }
    float attr_f(const char *k, float dflt) const { auto it = attrs.find(k); return it == attrs.end() ? dflt : it->second.f; }
    std::string attr_s(const char *k, const char *dflt) const { auto it = attrs.find(k); return it == attrs.end() ? dflt : it->second.s; }
    const std::vector<int64_t> *attr_ints(const char *k) const { auto it = attrs.find(k); return it == attrs.end() ? nullptr : &it->second.ints; }
    std::string input(size_t k) const { return k < in.size() ? in[k] : std::string(); }
};

struct ValueInfo { std::string name; int elem_type = 0; std::vector<int64_t> shape; };   // -1 = symbolic / unknown dimension

struct Graph {
    std::vector<Node> nodes;
    std::map<std::string, Tensor> init;
    std::vector<ValueInfo> inputs, outputs;
};

struct Model { int64_t ir_version = 0, opset = 0; Graph g; };

static void packed_i64(int wt, uint64_t val, const uint8_t *ptr, size_t len, std::vector<int64_t> &out, bool &ok)
{
    if (wt == 0) { out.push_back((int64_t)val); return; }
    Reader r(ptr, len);
    while (r.more()) { const uint64_t v = r.varint(); if (r.ok) out.push_back((int64_t)v); }
    ok = ok && r.ok;
}

static bool parse_tensor(const uint8_t *b, size_t n, Tensor &t)
{
    Reader r(b, n);
    int fno, wt; uint64_t val; const uint8_t *ptr; size_t len;
    bool ok = true;
    while (r.more() && r.field(fno, wt, val, ptr, len)) {
        switch (fno) {
        case 1: packed_i64(wt, val, ptr, len, t.dims, ok); break;
        case 2: t.dtype = (int)val; break;
        case 4:
            if (wt == 5) { float f; memcpy(&f, ptr, 4); t.fdata.push_back(f); }
            else if (wt == 2) { for (size_t i = 0; i + 4 <= len; i += 4) { float f; memcpy(&f, ptr + i, 4); t.fdata.push_back(f); } }
            break;
        case 5: case 7: packed_i64(wt, val, ptr, len, t.idata, ok); break;
        case 8: t.name.assign((const char *)ptr, len); break;
        case 9: t.has_raw = true; t.raw.assign((const char *)ptr, len); break;
        case 10:
            if (wt == 1) { double d; memcpy(&d, ptr, 8); t.ddata.push_back(d); }
            else if (wt == 2) { for (size_t i = 0; i + 8 <= len; i += 8) { double d; memcpy(&d, ptr + i, 8); t.ddata.push_back(d); } }
            break;
        case 14: if (val == 1) return false; break;      // external data
        default: break;
        }
    }
    if (t.dtype == DT_INT32)                              // int32_data travels as sign-extended varints
        for (auto &v : t.idata) v = (int64_t)(int32_t)v;
    return r.ok && ok;
}

static bool parse_attr(const uint8_t *b, size_t n, std::string &name, Attr &a)
{
    Reader r(b, n);
    int fno, wt; uint64_t val; const uint8_t *ptr; size_t len;
    bool ok = true;
    while (r.more() && r.field(fno, wt, val, ptr, len)) {
        switch (fno) {
        case 1: name.assign((const char *)ptr, len); break;
        case 2: { uint32_t v = (uint32_t)val; memcpy(&a.f, &v, 4); a.has_f = true; break; }
        case 3: a.i = (int64_t)val; a.has_i = true; break;
        case 4: a.s.assign((const char *)ptr, len); a.has_s = true; break;
        case 5: a.has_t = true; ok = ok && parse_tensor(ptr, len, a.t); break;
        case 7:
            if (wt == 5) { uint32_t v = (uint32_t)val; float f; memcpy(&f, &v, 4); a.floats.push_back(f); }
            else { for (size_t i = 0; i + 4 <= len; i += 4) { float f; memcpy(&f, ptr + i, 4); a.floats.push_back(f); } }
            break;
        case 8: packed_i64(wt, val, ptr, len, a.ints, ok); break;
        case 9: a.strings.emplace_back((const char *)ptr, len); break;
        case 20: a.type = (int)val; break;
        default: break;
        }
    }
    return r.ok && ok;
}

static bool parse_node(const uint8_t *b, size_t n, Node &nd)
{
    Reader r(b, n);
    int fno, wt; uint64_t val; const uint8_t *ptr; size_t len;
    bool ok = true;
    while (r.more() && r.field(fno, wt, val, ptr, len)) {
        switch (fno) {
        case 1: nd.in.emplace_back((const char *)ptr, len); break;
        case 2: nd.out.emplace_back((const char *)ptr, len); break;
        case 3: nd.name.assign((const char *)ptr, len); break;
        case 4: nd.op.assign((const char *)ptr, len); break;
        case 5: { std::string k; Attr a; ok = ok && parse_attr(ptr, len, k, a); nd.attrs[k] = a; break; }
        default: break;
        }
    }
    return r.ok && ok;
}

static bool parse_value_info(const uint8_t *b, size_t n, ValueInfo &vi)
{
    Reader r(b, n);
    int fno, wt; uint64_t val; const uint8_t *ptr; size_t len;
    while (r.more() && r.field(fno, wt, val, ptr, len)) {
        if (fno == 1) vi.name.assign((const char *)ptr, len);
        else if (fno == 2 && wt == 2) {                                  // TypeProto
            Reader r2(ptr, len);
            int f2, w2; uint64_t v2; const uint8_t *p2; size_t l2;
            while (r2.more() && r2.field(f2, w2, v2, p2, l2)) {
                if (f2 != 1 || w2 != 2) continue;                        // tensor_type
                Reader r3(p2, l2);
                int f3, w3; uint64_t v3; const uint8_t *p3; size_t l3;
                while (r3.more() && r3.field(f3, w3, v3, p3, l3)) {
                    if (f3 == 1) vi.elem_type = (int)v3;
                    else if (f3 == 2 && w3 == 2) {                       // TensorShapeProto
                        Reader r4(p3, l3);
                        int f4, w4; uint64_t v4; const uint8_t *p4; size_t l4;
                        while (r4.more() && r4.field(f4, w4, v4, p4, l4)) {
                            if (f4 != 1 || w4 != 2) continue;            // Dimension
                            int64_t d = -1;
                            Reader r5(p4, l4);
                            int f5, w5; uint64_t v5; const uint8_t *p5; size_t l5;
                            while (r5.more() && r5.field(f5, w5, v5, p5, l5))
                                if (f5 == 1) d = (int64_t)v5;
                            vi.shape.push_back(d);
                        }
                    }
                }
            }
        }
    }
    return r.ok;
}

static bool parse_graph(const uint8_t *b, size_t n, Graph &g)
{
    Reader r(b, n);
    int fno, wt; uint64_t val; const uint8_t *ptr; size_t len;
    bool ok = true;
    while (r.more() && r.field(fno, wt, val, ptr, len)) {
        if (wt != 2) continue;
        if (fno == 1) { g.nodes.emplace_back(); ok = ok && parse_node(ptr, len, g.nodes.back()); }
        else if (fno == 5) { Tensor t; ok = ok && parse_tensor(ptr, len, t); g.init[t.name] = std::move(t); }
        else if (fno == 11) { g.inputs.emplace_back(); ok = ok && parse_value_info(ptr, len, g.inputs.back()); }
        else if (fno == 12) { g.outputs.emplace_back(); ok = ok && parse_value_info(ptr, len, g.outputs.back()); }
    }
    // graph inputs that are really initialisers (IR < 4 style) are not runtime inputs
    std::vector<ValueInfo> real;
    for (auto &vi : g.inputs) if (!g.init.count(vi.name)) real.push_back(vi);
    g.inputs.swap(real);
    return r.ok && ok;
}

static bool parse_model(const uint8_t *b, size_t n, Model &m)
{
    Reader r(b, n);
    int fno, wt; uint64_t val; const uint8_t *ptr; size_t len;
    bool have_graph = false, ok = true;
    while (r.more() && r.field(fno, wt, val, ptr, len)) {
        if (fno == 1 && wt == 0) m.ir_version = (int64_t)val;
        else if (fno == 7 && wt == 2) { have_graph = true; ok = ok && parse_graph(ptr, len, m.g); }
        else if (fno == 8 && wt == 2) {
            Reader r2(ptr, len);
            int f2, w2; uint64_t v2; const uint8_t *p2; size_t l2;
            std::string dom; int64_t ver = 0;
            while (r2.more() && r2.field(f2, w2, v2, p2, l2)) {
                if (f2 == 1) dom.assign((const char *)p2, l2);
                else if (f2 == 2) ver = (int64_t)v2;
            }
            if (dom.empty() || dom == "ai.onnx") m.opset = ver;
        }
    }
    return r.ok && ok && have_graph;
}

// ------------------------------------------------------------------------------------------- probe evaluator (host, float64)
// Evaluates the small data-independent / map-only parts of the graph on probe inputs at load time: the adjacency
// normalisation, LSTM initial states, sequence_lens.  It never produces a score.
struct Val {
    std::vector<int64_t> shape;
    std::vector<double> v;
    int64_t numel() const { int64_t n = 1; for (auto d : shape) n *= d; return n; }
};

struct Evaluator {
    const Graph &g;
    std::map<std::string, const Node *> producer;
    std::map<std::string, Val> memo;
    std::string err;
    int depth = 0;
    explicit Evaluator(const Graph &gr) : g(gr)
    {
        for (auto &n : g.nodes) for (auto &o : n.out) if (!o.empty()) producer[o] = &n;
    }
    void feed(const std::string &name, const Val &v) { memo[name] = v; }
    bool fail(const std::string &m) { if (err.empty()) err = m; return false; }

    static bool broadcast(const Val &a, const Val &b, Val &out, const std::function<double(double, double)> &f)
    {
        const size_t r = std::max(a.shape.size(), b.shape.size());
        std::vector<int64_t> sa(r, 1), sb(r, 1);
        std::copy(a.shape.begin(), a.shape.end(), sa.begin() + (r - a.shape.size()));
        std::copy(b.shape.begin(), b.shape.end(), sb.begin() + (r - b.shape.size()));
        out.shape.resize(r);
        for (size_t i = 0; i < r; ++i) {
            if (sa[i] != sb[i] && sa[i] != 1 && sb[i] != 1) return false;
            out.shape[i] = std::max(sa[i], sb[i]);
        }
        const int64_t n = out.numel();
        out.v.resize((size_t)n);
        std::vector<int64_t> idx(r, 0);
        for (int64_t k = 0; k < n; ++k) {
            int64_t ia = 0, ib = 0;
            for (size_t i = 0; i < r; ++i) {
                ia = ia * sa[i] + (sa[i] == 1 ? 0 : idx[i]);
                ib = ib * sb[i] + (sb[i] == 1 ? 0 : idx[i]);
            }
            out.v[(size_t)k] = f(a.v[(size_t)ia], b.v[(size_t)ib]);
            for (int i = (int)r - 1; i >= 0; --i) { if (++idx[i] < out.shape[i]) break; idx[i] = 0; }
        }
        return true;
    }

    bool axes_of(const Node &n, size_t input_k, std::vector<int64_t> &axes, bool &present)
    {
        present = false;
        if (!n.input(input_k).empty()) {
            Val a;
            if (!eval(n.input(input_k), a)) return false;
            for (double d : a.v) axes.push_back((int64_t)d);
            present = true;
        } else if (auto *p = n.attr_ints("axes")) { axes = *p; present = true; }
        return true;
    }

    bool eval(const std::string &name, Val &out)
    {
        auto it = memo.find(name);
        if (it != memo.end()) { out = it->second; return true; }
        auto ci = g.init.find(name);
        if (ci != g.init.end()) {
            if (ci->second.numel() > (1 << 16)) return fail("probe evaluation reached the large initialiser '" + name + "'");
            Val v;
            v.shape = ci->second.dims;
            if (!ci->second.to_f64(v.v)) return fail("cannot decode initialiser '" + name + "'");
            memo[name] = v; out = v;
            return true;
        }
        auto pi = producer.find(name);
        if (pi == producer.end()) return fail("tensor '" + name + "' has no producer");
        if (++depth > 4000) return fail("graph too deep");
        const bool ok = eval_node(*pi->second);
        --depth;
        if (!ok) return false;
        it = memo.find(name);
        if (it == memo.end()) return fail("node '" + pi->second->name + "' did not produce '" + name + "'");
        out = it->second;
        return true;
    }

    bool eval_node(const Node &n)
    {
        const std::string &op = n.op;
        auto in = [&](size_t k, Val &v) { return eval(n.input(k), v); };
        Val a, b, y;
        if (op == "Add" || op == "Sub" || op == "Mul" || op == "Div") {
            if (!in(0, a) || !in(1, b)) return false;
            std::function<double(double, double)> f;
            if (op == "Add") f = [](double x, double z) { return x + z; };
            else if (op == "Sub") f = [](double x, double z) { return x - z; };
            else if (op == "Mul") f = [](double x, double z) { return x * z; };
            else f = [](double x, double z) { return x / z; };
            if (!broadcast(a, b, y, f)) return fail(op + " '" + n.name + "': shapes do not broadcast");
        } else if (op == "Sqrt" || op == "Reciprocal" || op == "Identity" || op == "Cast" || op == "Dropout" || op == "Relu" || op == "Neg") {
            if (!in(0, a)) return false;
            y = a;
            if (op == "Cast") {
                const int64_t to = n.attr_i("to", DT_FLOAT);
                if (to == DT_INT32 || to == DT_INT64 || to == DT_UINT8 || to == DT_INT8) for (auto &x : y.v) x = trunc(x);
                else if (to == DT_BOOL) for (auto &x : y.v) x = x != 0.0;
            }
            for (auto &x : y.v) {
                if (op == "Sqrt") x = sqrt(x);
                else if (op == "Reciprocal") x = 1.0 / x;
                else if (op == "Relu") x = x > 0 ? x : 0;
                else if (op == "Neg") x = -x;
            }
        } else if (op == "Constant") {
            auto it = n.attrs.find("value");
            if (it == n.attrs.end() || !it->second.has_t) return fail("Constant without a tensor value");
            y.shape = it->second.t.dims;
            if (!it->second.t.to_f64(y.v)) return fail("cannot decode Constant '" + n.name + "'");
        } else if (op == "Shape") {
            if (!in(0, a)) return false;
            y.shape = {(int64_t)a.shape.size()};
            for (auto d : a.shape) y.v.push_back((double)d);
        } else if (op == "Squeeze" || op == "Unsqueeze") {
            if (!in(0, a)) return false;
            std::vector<int64_t> axes; bool present;
            if (!axes_of(n, 1, axes, present)) return false;
            y = a;
            if (op == "Squeeze") {
                std::vector<int64_t> s;
                std::set<int64_t> ax;
                for (auto x : axes) ax.insert(x < 0 ? x + (int64_t)a.shape.size() : x);
                for (size_t i = 0; i < a.shape.size(); ++i) {
                    const bool drop = present ? ax.count((int64_t)i) > 0 : a.shape[i] == 1;
                    if (drop && a.shape[i] != 1) return fail("Squeeze of a non-unit axis");
                    if (!drop) s.push_back(a.shape[i]);
                }
                y.shape = s;
            } else {
                if (!present) return fail("Unsqueeze without axes");
                const int64_t r = (int64_t)a.shape.size() + (int64_t)axes.size();
                std::set<int64_t> ax;
                for (auto x : axes) ax.insert(x < 0 ? x + r : x);
                std::vector<int64_t> s;
                size_t k = 0;
                for (int64_t i = 0; i < r; ++i) s.push_back(ax.count(i) ? 1 : a.shape[k++]);
                y.shape = s;
            }
        } else if (op == "Reshape" || op == "Expand" || op == "ConstantOfShape" || op == "Tile") {
            Val s;
            if (op == "ConstantOfShape") {
                if (!in(0, s)) return false;
                double fill = 0.0;
                auto it = n.attrs.find("value");
                if (it != n.attrs.end() && it->second.has_t) { std::vector<double> t; if (!it->second.t.to_f64(t) || t.empty()) return fail("ConstantOfShape value"); fill = t[0]; }
                for (double d : s.v) y.shape.push_back((int64_t)d);
                y.v.assign((size_t)y.numel(), fill);
            } else {
                if (!in(0, a) || !in(1, s)) return false;
                if (op == "Reshape") {
                    int64_t known = 1, infer = -1;
                    for (size_t i = 0; i < s.v.size(); ++i) {
                        int64_t d = (int64_t)s.v[i];
                        if (d == 0) d = i < a.shape.size() ? a.shape[i] : 1;
                        if (d == -1) infer = (int64_t)i; else known *= d;
                        y.shape.push_back(d);
                    }
                    if (infer >= 0) y.shape[(size_t)infer] = known ? a.numel() / known : 0;
                    if (y.numel() != a.numel()) return fail("Reshape changes the element count");
                    y.v = a.v;
                } else if (op == "Expand") {
                    Val ones;
                    for (double d : s.v) ones.shape.push_back((int64_t)d);
                    ones.v.assign((size_t)ones.numel(), 0.0);
                    if (!broadcast(a, ones, y, [](double x, double) { return x; })) return fail("Expand shapes");
                } else {
                    if (s.v.size() != a.shape.size()) return fail("Tile repeats rank");
                    y.shape = a.shape;
                    for (size_t i = 0; i < s.v.size(); ++i) y.shape[i] *= (int64_t)s.v[i];
                    const int64_t nn = y.numel();
                    y.v.resize((size_t)nn);
                    std::vector<int64_t> idx(y.shape.size(), 0);
                    for (int64_t k = 0; k < nn; ++k) {
                        int64_t ia = 0;
                        for (size_t i = 0; i < idx.size(); ++i) ia = ia * a.shape[i] + idx[i] % a.shape[i];
                        y.v[(size_t)k] = a.v[(size_t)ia];
                        for (int i = (int)idx.size() - 1; i >= 0; --i) { if (++idx[i] < y.shape[i]) break; idx[i] = 0; }
                    }
                }
            }
        } else if (op == "EyeLike") {
            if (!in(0, a)) return false;
            if (a.shape.size() != 2) return fail("EyeLike of a non-matrix");
            const int64_t k = n.attr_i("k", 0);
            y.shape = a.shape;
            y.v.assign((size_t)y.numel(), 0.0);
            for (int64_t i = 0; i < a.shape[0]; ++i) if (i + k >= 0 && i + k < a.shape[1]) y.v[(size_t)(i * a.shape[1] + i + k)] = 1.0;
        } else if (op == "Transpose") {
            if (!in(0, a)) return false;
            const size_t r = a.shape.size();
            std::vector<int64_t> perm;
            if (auto *p = n.attr_ints("perm")) perm = *p; else for (size_t i = 0; i < r; ++i) perm.push_back((int64_t)(r - 1 - i));
            if (perm.size() != r) return fail("Transpose perm rank");
            y.shape.resize(r);
            for (size_t i = 0; i < r; ++i) y.shape[i] = a.shape[(size_t)perm[i]];
            std::vector<int64_t> stride(r, 1);
            for (int i = (int)r - 2; i >= 0; --i) stride[(size_t)i] = stride[(size_t)i + 1] * a.shape[(size_t)i + 1];
            const int64_t nn = y.numel();
            y.v.resize((size_t)nn);
            std::vector<int64_t> idx(r, 0);
            for (int64_t k = 0; k < nn; ++k) {
                int64_t ia = 0;
                for (size_t i = 0; i < r; ++i) ia += idx[i] * stride[(size_t)perm[i]];
                y.v[(size_t)k] = a.v[(size_t)ia];
                for (int i = (int)r - 1; i >= 0; --i) { if (++idx[(size_t)i] < y.shape[(size_t)i]) break; idx[(size_t)i] = 0; }
            }
        } else if (op == "ReduceSum" || op == "ReduceMax") {
            if (!in(0, a)) return false;
            std::vector<int64_t> axes; bool present;
            if (!axes_of(n, 1, axes, present)) return false;
            const bool keep = n.attr_i("keepdims", 1) != 0;
            const size_t r = a.shape.size();
            std::vector<bool> red(r, !present);
            for (auto x : axes) red[(size_t)(x < 0 ? x + (int64_t)r : x)] = true;
            std::vector<int64_t> os(r);
            for (size_t i = 0; i < r; ++i) os[i] = red[i] ? 1 : a.shape[i];
            Val t;
            t.shape = os;
            t.v.assign((size_t)t.numel(), op == "ReduceSum" ? 0.0 : -INFINITY);
            std::vector<int64_t> idx(r, 0);
            for (int64_t k = 0; k < a.numel(); ++k) {
                int64_t io = 0;
                for (size_t i = 0; i < r; ++i) io = io * os[i] + (red[i] ? 0 : idx[i]);
                if (op == "ReduceSum") t.v[(size_t)io] += a.v[(size_t)k]; else t.v[(size_t)io] = std::max(t.v[(size_t)io], a.v[(size_t)k]);
                for (int i = (int)r - 1; i >= 0; --i) { if (++idx[(size_t)i] < a.shape[(size_t)i]) break; idx[(size_t)i] = 0; }
            }
            y.v = t.v;
            for (size_t i = 0; i < r; ++i) if (keep || !red[i]) y.shape.push_back(os[i]);
        } else if (op == "MatMul") {
            if (!in(0, a) || !in(1, b)) return false;
            if (a.shape.size() < 2 || b.shape.size() < 2) return fail("MatMul of vectors is not supported by the probe evaluator");
            const int64_t M = a.shape[a.shape.size() - 2], K = a.shape.back(), K2 = b.shape[b.shape.size() - 2], N = b.shape.back();
            if (K != K2) return fail("MatMul '" + n.name + "': inner dimensions differ");
            int64_t ba = a.numel() / (M * K), bb = b.numel() / (K * N);
            if (ba != bb && ba != 1 && bb != 1) return fail("MatMul batch broadcast");
            const int64_t B = std::max(ba, bb);
            y.shape = ba >= bb ? a.shape : b.shape;
            y.shape[y.shape.size() - 2] = M; y.shape.back() = N;
            y.v.assign((size_t)(B * M * N), 0.0);
            for (int64_t q = 0; q < B; ++q) {
                const double *pa = a.v.data() + (ba == 1 ? 0 : q) * M * K, *pb = b.v.data() + (bb == 1 ? 0 : q) * K * N;
                double *py = y.v.data() + q * M * N;
                for (int64_t i = 0; i < M; ++i) for (int64_t k = 0; k < K; ++k) { const double x = pa[i * K + k]; for (int64_t j = 0; j < N; ++j) py[i * N + j] += x * pb[k * N + j]; }
            }
        } else if (op == "Gather") {
            Val idx;
            if (!in(0, a) || !in(1, idx)) return false;
            if (a.shape.size() != 1 || n.attr_i("axis", 0) != 0) return fail("Gather: only 1-D sources");
            y.shape = idx.shape;
            for (double d : idx.v) { int64_t i = (int64_t)d; if (i < 0) i += a.shape[0]; if (i < 0 || i >= a.shape[0]) return fail("Gather index"); y.v.push_back(a.v[(size_t)i]); }
        } else if (op == "Concat") {
            const int64_t axis = n.attr_i("axis", 0);
            std::vector<Val> parts(n.in.size());
            for (size_t k = 0; k < n.in.size(); ++k) if (!in(k, parts[k])) return false;
            if (parts.empty() || parts[0].shape.size() != 1 || (axis != 0 && axis != -1)) return fail("Concat: only 1-D tensors");
            for (auto &p : parts) y.v.insert(y.v.end(), p.v.begin(), p.v.end());
            y.shape = {(int64_t)y.v.size()};
        } else if (op == "Slice") {
            Val st, en;
            if (!in(0, a) || !in(1, st) || !in(2, en)) return false;
            if (a.shape.size() != 1 || st.v.size() != 1) return fail("Slice: only 1-D tensors");
            int64_t s0 = (int64_t)st.v[0], e0 = (int64_t)std::min(en.v[0], 1e15), L = a.shape[0];
            if (s0 < 0) s0 += L;
            if (e0 < 0) e0 += L;
            s0 = std::max<int64_t>(0, std::min(L, s0)); e0 = std::max<int64_t>(0, std::min(L, e0));
            if (!n.input(4).empty()) { Val sp; if (!in(4, sp)) return false; if (sp.v.size() != 1 || sp.v[0] != 1.0) return fail("Slice step"); }
            for (int64_t i = s0; i < e0; ++i) y.v.push_back(a.v[(size_t)i]);
            y.shape = {(int64_t)y.v.size()};
        } else {
            return fail("operator " + op + " ('" + n.name + "') is not supported by the load-time probe evaluator");
        }
        memo[n.out[0]] = y;
        return true;
    }
};

// ------------------------------------------------------------------------------------------- recogniser
struct Plan {
    bool is_cnn = false;
    std::vector<std::string> input_names;
    std::string error;
    // GCN
    int H = 0, E = 0, F = 0, C = 0, act = 0;
    float alpha = 1.f, eps = 0.f;
    std::vector<std::vector<float>> lstm_W, lstm_R, lstm_B;     // B empty = none
    std::vector<float> aa_W, lm_W, lm_b, fc_W, fc_b, out_W, out_b;
    std::vector<std::vector<float>> gc_W, gc_b;
    std::vector<int> gc_dims;
    std::map<std::string, std::string> roles;                   // role -> initialiser name
    // CNN
    std::vector<std::vector<float>> conv_W;                     // [F, 26, w] each
    std::vector<int> conv_filters, conv_width, conv_pad_left;
    std::vector<float> scale, shift;
    unsigned long long lm_hash = 0;
};

static const std::set<std::string> kShapeOps = {"Transpose", "Squeeze", "Unsqueeze", "Reshape", "Identity", "Dropout", "Cast", "Flatten"};

struct GraphIndex {
    const Graph &g;
    std::map<std::string, const Node *> producer;
    std::map<std::string, std::vector<const Node *>> consumers;
    std::map<std::string, const Tensor *> cst;                  // initialisers + Constant nodes
    explicit GraphIndex(const Graph &gr) : g(gr)
    {
        for (auto &kv : g.init) cst[kv.first] = &kv.second;
        for (auto &n : g.nodes) {
            for (auto &o : n.out) if (!o.empty()) producer[o] = &n;
            for (auto &i : n.in) if (!i.empty()) consumers[i].push_back(&n);
            if (n.op == "Constant") { auto it = n.attrs.find("value"); if (it != n.attrs.end() && it->second.has_t && !n.out.empty()) cst[n.out[0]] = &it->second.t; }
        }
    }
    bool is_const(const std::string &t) const { return cst.count(t) > 0; }
    std::string back(std::string t) const
    {
        for (;;) {
            auto it = producer.find(t);
            if (it == producer.end() || !kShapeOps.count(it->second->op)) return t;
            t = it->second->in.empty() ? std::string() : it->second->in[0];
        }
    }
    void fwd(const std::string &t, std::vector<const Node *> &out) const
    {
        auto it = consumers.find(t);
        if (it == consumers.end()) return;
        for (auto *n : it->second) {
            if (kShapeOps.count(n->op)) { if (!n->out.empty()) fwd(n->out[0], out); }
            else out.push_back(n);
        }
    }
    std::vector<const Node *> fwd(const std::string &t) const { std::vector<const Node *> o; fwd(t, o); return o; }
};

static std::string fmt(const char *f, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, f);
    vsnprintf(buf, sizeof buf, f, ap);
    va_end(ap);
    return buf;
}

static std::string dims_str(const Tensor &t)
{
    std::string s = "(";
    for (size_t i = 0; i < t.dims.size(); ++i) s += (i ? ", " : "") + std::to_string(t.dims[i]);
    return s + ")";
}

// constant-weight product node: MatMul with a constant right operand, or Gemm (tf2onnx fuses MatMul + Add on 2-D inputs)
struct Dense {
    const Node *node = nullptr;
    std::string wname;
    int rows = 0, cols = 0;
    std::vector<float> W;        // [rows, cols] row-major (Gemm transB undone)
    std::vector<float> bias;     // Gemm C, or the Add that follows
    std::string bias_name, out;  // tensor after the optional bias
};

static bool dense_bias_after(const GraphIndex &ix, Dense &d)
{
    d.out = d.node->out[0];
    if (!d.bias.empty()) return true;
    for (auto *c : ix.fwd(d.out)) {
        if (c->op != "Add") continue;
        std::vector<std::string> k;
        for (auto &i : c->in) if (ix.is_const(i)) k.push_back(i);
        if (k.size() != 1) continue;
        const Tensor *t = ix.cst.at(k[0]);
        if (t->dims.empty() || t->numel() != t->dims.back()) continue;          // [N] or [1, .., N]
        if (!t->to_f32(d.bias)) return false;
        d.bias_name = k[0];
        d.out = c->out[0];
        return true;
    }
    return true;
}

#define PLAN_FAIL(...) do { plan.error = std::string(kind) + fmt(__VA_ARGS__); return false; } while (0)

static bool recognise_gcn(const Model &m, Plan &plan)
{
    static const char *kind = "ONNX graph is not a supported DeepFRI GCN head: ";
    const Graph &g = m.g;
    GraphIndex ix(g);
    if (g.inputs.size() != 2) PLAN_FAIL("expected 2 inputs (cmap, seq), found %zu", g.inputs.size());
    int seq_i = -1;
    for (int i = 0; i < 2; ++i)
        if (g.inputs[i].shape.size() == 3 && g.inputs[i].shape[2] == 26) { if (seq_i >= 0) seq_i = -2; else seq_i = i; }
    if (seq_i < 0) PLAN_FAIL("cannot identify the [batch, L, 26] one-hot sequence input");
    if (seq_i != 1) PLAN_FAIL("inputs must be ordered (cmap, seq) as the reference feeds them (predict.pyx:87-90)");
    const std::string seq_name = g.inputs[1].name, cmap_name = g.inputs[0].name;
    plan.input_names = {cmap_name, seq_name};

    // roles a tensor depends on: bit 0 seq, bit 1 cmap, bit 2 lstm
    std::map<std::string, int> memo;
    std::function<int(const std::string &)> deps = [&](const std::string &t) -> int {
        auto it = memo.find(t);
        if (it != memo.end()) return it->second;
        memo[t] = 0;
        int d = 0;
        if (t == seq_name) d = 1;
        else if (t == cmap_name) d = 2;
        else {
            auto p = ix.producer.find(t);
            if (p != ix.producer.end()) {
                if (p->second->op == "LSTM") d |= 4;
                for (auto &i : p->second->in) if (!i.empty() && !ix.is_const(i)) d |= deps(i);
            }
        }
        memo[t] = d;
        return d;
    };

    // ---- LSTM stack
    std::vector<const Node *> lstms;
    for (auto &n : g.nodes) if (n.op == "LSTM") lstms.push_back(&n);
    if (lstms.empty()) PLAN_FAIL("no LSTM language-model layers found");
    const int H = (int)lstms[0]->attr_i("hidden_size", 0);
    const Node *prev = nullptr;
    for (size_t k = 0; k < lstms.size(); ++k) {
        const Node *n = lstms[k];
        if (n->attr_s("direction", "forward") != "forward" || n->attr_i("layout", 0) != 0) PLAN_FAIL("only forward, layout-0 LSTM layers are supported");
        auto act = n->attrs.find("activations");
        if (act != n->attrs.end()) {
            std::vector<std::string> a = act->second.strings;
            for (auto &s : a) for (auto &c : s) c = (char)tolower(c);
            if (a != std::vector<std::string>{"sigmoid", "tanh", "tanh"}) PLAN_FAIL("LSTM uses non-default activations");
        }
        if (n->attrs.count("clip") || n->attr_i("input_forget", 0) != 0) PLAN_FAIL("LSTM with clip / input_forget is not supported");
        if ((int)n->attr_i("hidden_size", 0) != H) PLAN_FAIL("stacked LSTM layers have different hidden sizes");
        if (!n->input(7).empty()) PLAN_FAIL("LSTM with peepholes is not supported");
        const std::string src = ix.back(n->input(0));
        if (k == 0 && src != seq_name) PLAN_FAIL("first LSTM layer is not fed by the sequence input");
        if (k > 0) { auto p = ix.producer.find(src); if (p == ix.producer.end() || p->second != prev) PLAN_FAIL("LSTM layers are not stacked"); }
        auto W = ix.cst.find(n->input(1)), R = ix.cst.find(n->input(2));
        if (W == ix.cst.end() || R == ix.cst.end()) PLAN_FAIL("LSTM weights are not constant initialisers");
        const int in_dim = k == 0 ? 26 : H;
        const std::vector<int64_t> ws = {1, 4 * H, in_dim}, rs = {1, 4 * H, H}, bs = {1, 8 * H};
        if (W->second->dims != ws || R->second->dims != rs)
            PLAN_FAIL("LSTM layer %zu: unexpected weight shapes W%s R%s", k + 1, dims_str(*W->second).c_str(), dims_str(*R->second).c_str());
        plan.lstm_W.emplace_back(); plan.lstm_R.emplace_back(); plan.lstm_B.emplace_back();
        if (!W->second->to_f32(plan.lstm_W.back()) || !R->second->to_f32(plan.lstm_R.back())) PLAN_FAIL("cannot decode LSTM weights");
        plan.roles[fmt("lstm%zu_W", k + 1)] = n->input(1);
        plan.roles[fmt("lstm%zu_R", k + 1)] = n->input(2);
        if (!n->input(3).empty()) {
            auto B = ix.cst.find(n->input(3));
            if (B == ix.cst.end() || B->second->dims != bs) PLAN_FAIL("LSTM layer %zu: bias is not a constant [1, 8H] tensor", k + 1);
            if (!B->second->to_f32(plan.lstm_B.back())) PLAN_FAIL("cannot decode LSTM bias");
            plan.roles[fmt("lstm%zu_B", k + 1)] = n->input(3);
        }
        prev = n;
    }
    // sequence_lens / initial states: accepted when they are what the fused kernel assumes (full length, zeros) - checked on probes
    for (int probe_L : {7, 11}) {
        Evaluator ev(g);
        Val s; s.shape = {1, probe_L, 26}; s.v.assign((size_t)probe_L * 26, 0.0);
        for (int i = 0; i < probe_L; ++i) s.v[(size_t)i * 26 + (i * 5 + 3) % 26] = 1.0;
        ev.feed(seq_name, s);
        Val c; c.shape = {1, probe_L, probe_L}; c.v.assign((size_t)probe_L * probe_L, 0.0);
        ev.feed(cmap_name, c);
        for (auto *n : lstms) {
            if (!n->input(4).empty()) {
                Val v;
                if (!ev.eval(n->input(4), v)) PLAN_FAIL("cannot verify LSTM sequence_lens: %s", ev.err.c_str());
                for (double x : v.v) if ((int)x != probe_L) PLAN_FAIL("LSTM sequence_lens is not the full sequence length");
            }
            for (int k : {5, 6}) {
                if (n->input((size_t)k).empty()) continue;
                Val v;
                if (!ev.eval(n->input((size_t)k), v)) PLAN_FAIL("cannot verify LSTM initial state: %s", ev.err.c_str());
                for (double x : v.v) if (x != 0.0) PLAN_FAIL("LSTM with a non-zero initial state is not supported");
            }
        }
    }

    // ---- products with a constant weight, classified by what they depend on; data x data MatMuls
    auto ancestors_have_reducesum = [&](const std::string &t) {
        std::vector<std::string> stack = {t};
        std::set<std::string> seen;
        while (!stack.empty()) {
            std::string x = stack.back(); stack.pop_back();
            if (seen.count(x)) continue;
            seen.insert(x);
            auto p = ix.producer.find(x);
            if (p == ix.producer.end()) continue;
            if (p->second->op == "MatMul" || p->second->op == "Gemm") continue;
            if (p->second->op == "ReduceSum") return true;
            for (auto &i : p->second->in) if (!i.empty() && !ix.is_const(i)) stack.push_back(i);
        }
        return false;
    };
    std::vector<Dense> gcs, heads;
    Dense aa, lm;
    std::vector<const Node *> adj_products;
    for (auto &n : g.nodes) {
        if (n.op != "MatMul" && n.op != "Gemm") continue;
        const bool c0 = ix.is_const(n.input(0)), c1 = ix.is_const(n.input(1));
        if (!c0 && !c1) {
            if (n.op == "Gemm") PLAN_FAIL("Gemm '%s' with two data operands", n.name.c_str());
            const int d0 = deps(n.input(0)), d1 = deps(n.input(1));
            if (d0 == 2 && d1 == 2) continue;                                  // inside the adjacency normalisation
            if (d0 == 2 && (d1 & 1)) { adj_products.push_back(&n); continue; } // A_norm . X
            PLAN_FAIL("MatMul '%s' multiplies two data tensors but is not an adjacency product (A_norm on the left)", n.name.c_str());
        }
        if (c0 || !c1) PLAN_FAIL("%s '%s': the weight must be the right operand", n.op.c_str(), n.name.c_str());
        Dense d;
        d.node = &n;
        d.wname = n.input(1);
        const Tensor *w = ix.cst.at(d.wname);
        if (w->dims.size() != 2) PLAN_FAIL("%s '%s': weight rank %zu", n.op.c_str(), n.name.c_str(), w->dims.size());
        std::vector<float> raw;
        if (!w->to_f32(raw)) PLAN_FAIL("cannot decode weight '%s'", d.wname.c_str());
        d.rows = (int)w->dims[0]; d.cols = (int)w->dims[1];
        d.W = raw;
        if (n.op == "Gemm") {
            if (n.attr_i("transA", 0) || n.attr_f("alpha", 1.f) != 1.f || n.attr_f("beta", 1.f) != 1.f) PLAN_FAIL("Gemm '%s' with transA / alpha / beta", n.name.c_str());
            if (n.attr_i("transB", 0)) {
                std::swap(d.rows, d.cols);
                for (int r = 0; r < d.rows; ++r) for (int c = 0; c < d.cols; ++c) d.W[(size_t)r * d.cols + c] = raw[(size_t)c * d.rows + r];
            }
            if (!n.input(2).empty()) {
                auto b = ix.cst.find(n.input(2));
                if (b == ix.cst.end() || b->second->numel() != d.cols || !b->second->to_f32(d.bias)) PLAN_FAIL("Gemm '%s': bias is not a constant [N] tensor", n.name.c_str());
                d.bias_name = n.input(2);
            }
        }
        const int dp = deps(n.input(0));
        if (!(dp & 2) && !(dp & 4) && (dp & 1)) { if (aa.node) PLAN_FAIL("more than one sequence embedding MatMul"); aa = d; }
        else if (!(dp & 2) && (dp & 4)) { if (lm.node) PLAN_FAIL("more than one language-model embedding MatMul"); lm = d; }
        else if (dp & 2) { if (!heads.empty() || ancestors_have_reducesum(n.input(0))) heads.push_back(d); else gcs.push_back(d); }
        else PLAN_FAIL("%s '%s' has no recognised role", n.op.c_str(), n.name.c_str());
    }
    if (!aa.node || !lm.node) PLAN_FAIL("embedding layers (AA_embedding / LM_embedding) not found");
    if (aa.rows != 26 || lm.rows != H || aa.cols != lm.cols) PLAN_FAIL("embedding shapes (%d, %d) / (%d, %d) are inconsistent", aa.rows, aa.cols, lm.rows, lm.cols);
    const int E = aa.cols;
    if (!dense_bias_after(ix, lm) || !dense_bias_after(ix, aa)) PLAN_FAIL("cannot decode an embedding bias");
    if (!aa.bias.empty()) PLAN_FAIL("AA_embedding with a bias is not supported");
    if (gcs.empty() || adj_products.size() != gcs.size())
        PLAN_FAIL("found %zu GraphConv weight MatMuls but %zu adjacency products", gcs.size(), adj_products.size());
    if (heads.size() != 2) PLAN_FAIL("expected dense + output layers after pooling, found %zu MatMuls", heads.size());
    // the embedding sum and its ReLU
    {
        bool relu = false, summed = false;
        for (auto *c : ix.fwd(lm.out)) {
            if (c->op != "Add") continue;
            bool other = false;
            for (auto &i : c->in) if (ix.back(i) == aa.out || i == aa.out) other = true;
            if (!other) continue;
            summed = true;
            for (auto *r : ix.fwd(c->out[0])) if (r->op == "Relu") relu = true;
        }
        if (!summed) PLAN_FAIL("LM_embedding and AA_embedding are not summed");
        if (!relu) PLAN_FAIL("embedding sum is not followed by ReLU");
    }
    // ---- GraphConv stack
    int width = E;
    std::set<int> acts;
    std::set<float> alphas;
    for (size_t k = 0; k < gcs.size(); ++k) {
        Dense &d = gcs[k];
        if (d.rows != width) PLAN_FAIL("GraphConv layer %zu: weight (%d, %d) does not follow width %d", k + 1, d.rows, d.cols, width);
        if (!dense_bias_after(ix, d)) PLAN_FAIL("cannot decode a GraphConv bias");
        int act = 0; float alpha = 1.f;
        std::string cur = d.out;
        for (int hop = 0; hop < 3; ++hop) {                 // activation directly after (A.X).W, or after the adjacency product of A.(X.W)
            auto nxt = ix.fwd(cur);
            const Node *hit = nullptr, *mm = nullptr;
            for (auto *c : nxt) { if (c->op == "Relu" || c->op == "Elu") hit = hit ? hit : c; }
            if (hit) { act = hit->op == "Relu" ? 1 : 2; alpha = hit->attr_f("alpha", 1.f); break; }
            for (auto *c : nxt) if (c->op == "MatMul" && !ix.is_const(c->input(0)) && !ix.is_const(c->input(1))) mm = mm ? mm : c;
            if (!mm) break;
            cur = mm->out[0];
        }
        acts.insert(act); alphas.insert(alpha);
        plan.gc_W.push_back(d.W); plan.gc_b.push_back(d.bias); plan.gc_dims.push_back(d.cols);
        plan.roles[fmt("gc%zu_W", k + 1)] = d.wname;
        if (!d.bias_name.empty()) plan.roles[fmt("gc%zu_b", k + 1)] = d.bias_name;
        width = d.cols;
    }
    if (acts.size() != 1 || alphas.size() != 1) PLAN_FAIL("GraphConv layers use different activations");
    plan.act = *acts.begin(); plan.alpha = *alphas.begin();
    int G = 0;
    for (int d : plan.gc_dims) G += d;
    Dense &fc = heads[0], &out = heads[1];
    if (fc.rows != G) PLAN_FAIL("dense layer expects %d pooled features, GraphConv stack gives %d (per-layer outputs must be concatenated)", fc.rows, G);
    if (!dense_bias_after(ix, fc) || !dense_bias_after(ix, out)) PLAN_FAIL("cannot decode a head bias");
    {
        bool relu = false;
        for (auto *c : ix.fwd(fc.out)) if (c->op == "Relu") relu = true;
        if (!relu) PLAN_FAIL("dense layer after pooling is not followed by ReLU");
    }
    if (out.rows != fc.cols || out.cols % 2) PLAN_FAIL("output layer weight (%d, %d) inconsistent", out.rows, out.cols);
    std::vector<const Node *> sm;
    for (auto &n : g.nodes) if (n.op == "Softmax") sm.push_back(&n);
    if (sm.size() != 1 || g.outputs.empty() || sm[0]->out[0] != g.outputs[0].name) PLAN_FAIL("graph does not end in a single Softmax");
    { const int64_t ax = sm[0]->attr_i("axis", -1); if (ax != -1 && ax != 2) PLAN_FAIL("Softmax is not over the last axis"); }

    // ---- degree normalisation: epsilon = the scalar added to sqrt(rowsum); then the whole sub-graph is verified on probes
    bool have_eps = false;
    for (auto &n : g.nodes) {
        if (n.op != "Sqrt" || deps(n.input(0)) != 2) continue;
        for (auto *c : ix.fwd(n.out[0])) {
            if (c->op != "Add") continue;
            for (auto &i : c->in) {
                auto k = ix.cst.find(i);
                if (k == ix.cst.end() || k->second->numel() != 1) continue;
                std::vector<float> v;
                if (!k->second->to_f32(v)) continue;
                if (have_eps && v[0] != plan.eps) PLAN_FAIL("GraphConv layers use different normalisation epsilons");
                plan.eps = v[0]; have_eps = true;
            }
        }
    }
    if (!have_eps) PLAN_FAIL("degree normalisation (1 / (eps + sqrt(rowsum))) not found");
    for (int L : {6, 9}) {
        Evaluator ev(g);
        Val A; A.shape = {1, L, L}; A.v.assign((size_t)L * L, 0.0);
        unsigned s = 12345u + (unsigned)L;
        for (int i = 0; i < L; ++i) for (int j = 0; j < L; ++j) { s = s * 1664525u + 1013904223u; A.v[(size_t)i * L + j] = ((s >> 16) & 3) == 0 ? 1.0 : 0.0; }
        A.v[0] = 1.0; A.v[(size_t)L + 1] = 0.0; A.v[(size_t)2 * L + 2] = 1.0;                 // diagonal both set and unset
        A.v[(size_t)1 * L + 4] = 1.0; A.v[(size_t)4 * L + 1] = 0.0;                             // certainly non-symmetric
        ev.feed(cmap_name, A);
        std::vector<double> Ah(A.v), d((size_t)L);
        for (int i = 0; i < L; ++i) Ah[(size_t)i * L + i] = 1.0;
        for (int i = 0; i < L; ++i) { double r = 0; for (int j = 0; j < L; ++j) r += Ah[(size_t)i * L + j]; d[(size_t)i] = 1.0 / ((double)plan.eps + sqrt(r)); }
        for (auto *mmn : adj_products) {
            Val got;
            if (!ev.eval(mmn->input(0), got)) PLAN_FAIL("cannot verify the adjacency normalisation feeding '%s': %s", mmn->name.c_str(), ev.err.c_str());
            if (got.numel() != (int64_t)L * L) PLAN_FAIL("adjacency operand of '%s' is not [1, L, L]", mmn->name.c_str());
            for (int i = 0; i < L; ++i) for (int j = 0; j < L; ++j) {
                const double want = d[(size_t)i] * Ah[(size_t)i * L + j] * d[(size_t)j];
                if (fabs(got.v[(size_t)i * L + j] - want) > 1e-9)
                    PLAN_FAIL("the adjacency operand of '%s' is not D (A - diag(A) + I) D with d = 1 / (eps + sqrt(rowsum)): entry (%d, %d) of a %d-residue "
                              "probe is %.9g, expected %.9g", mmn->name.c_str(), i, j, L, got.v[(size_t)i * L + j], want);
            }
        }
    }

    plan.H = H; plan.E = E; plan.F = fc.cols; plan.C = out.cols / 2;
    plan.aa_W = aa.W; plan.lm_W = lm.W; plan.lm_b = lm.bias;
    plan.fc_W = fc.W; plan.fc_b = fc.bias; plan.out_W = out.W; plan.out_b = out.bias;
    plan.roles["aa_W"] = aa.wname; plan.roles["lm_W"] = lm.wname;
    if (!lm.bias_name.empty()) plan.roles["lm_b"] = lm.bias_name;
    plan.roles["fc_W"] = fc.wname; plan.roles["out_W"] = out.wname;
    if (!fc.bias_name.empty()) plan.roles["fc_b"] = fc.bias_name;
    if (!out.bias_name.empty()) plan.roles["out_b"] = out.bias_name;
    unsigned long long h = 1469598103934665603ull;
    auto mix = [&](const std::vector<float> &v) { const unsigned char *p = (const unsigned char *)v.data(); for (size_t i = 0; i < v.size() * 4; ++i) { h ^= p[i]; h *= 1099511628211ull; } };
    for (auto &v : plan.lstm_W) mix(v);
    for (auto &v : plan.lstm_R) mix(v);
    for (auto &v : plan.lstm_B) mix(v);
    plan.lm_hash = h;
    return true;
}

static bool recognise_cnn(const Model &m, Plan &plan)
{
    static const char *kind = "ONNX graph is not a supported DeepCNN head: ";
    const Graph &g = m.g;
    GraphIndex ix(g);
    plan.is_cnn = true;
    if (g.inputs.size() != 1) PLAN_FAIL("expected the one-hot sequence as the single input, found %zu inputs", g.inputs.size());
    const ValueInfo &vi = g.inputs[0];
    if (vi.shape.size() != 3 || vi.shape[2] != 26) PLAN_FAIL("input '%s' is not [batch, L, 26]", vi.name.c_str());
    const std::string seq_name = vi.name;
    plan.input_names = {seq_name};
    static const std::set<std::string> allowed = {"Conv", "Concat", "BatchNormalization", "Relu", "ReduceMax", "GlobalMaxPool", "MatMul", "Gemm", "Add",
                                                  "Softmax", "Constant"};
    for (auto &n : g.nodes)
        if (!allowed.count(n.op) && !kShapeOps.count(n.op))
            PLAN_FAIL("unexpected operator %s ('%s'); a language-model DeepCNN variant is not supported", n.op.c_str(), n.name.c_str());
    struct ConvInfo { std::vector<float> W; int F, w, pl; std::vector<float> b; std::string wname; };
    std::map<std::string, ConvInfo> info;
    std::vector<const Node *> convs;
    for (auto &n : g.nodes) if (n.op == "Conv") convs.push_back(&n);
    if (convs.empty()) PLAN_FAIL("no Conv layers found");
    for (auto *n : convs) {
        if (ix.back(n->input(0)) != seq_name) PLAN_FAIL("Conv '%s' is not fed by the sequence input", n->name.c_str());
        auto Wt = ix.cst.find(n->input(1));
        if (Wt == ix.cst.end()) PLAN_FAIL("Conv '%s': weights are not constant", n->name.c_str());
        const Tensor &W = *Wt->second;
        bool two_d;
        if (W.dims.size() == 4 && W.dims[2] == 1) two_d = true;
        else if (W.dims.size() == 3) two_d = false;
        else PLAN_FAIL("Conv '%s': weight shape %s is not [F, 26, 1, w] / [F, 26, w]", n->name.c_str(), dims_str(W).c_str());
        ConvInfo ci;
        ci.F = (int)W.dims[0]; ci.w = (int)W.dims.back();
        if (W.dims[1] != 26) PLAN_FAIL("Conv '%s': %lld input channels", n->name.c_str(), (long long)W.dims[1]);
        auto all_one = [&](const char *k) { auto *p = n->attr_ints(k); if (!p) return true; for (auto v : *p) if (v != 1) return false; return true; };
        if (n->attr_i("group", 1) != 1 || !all_one("strides") || !all_one("dilations")) PLAN_FAIL("Conv '%s': only group 1 / stride 1 / dilation 1", n->name.c_str());
        const std::string autop = n->attr_s("auto_pad", "NOTSET");
        int pl, pr;
        const int k = ci.w;
        if (autop == "SAME_UPPER") { pl = (k - 1) / 2; pr = k - 1 - pl; }
        else if (autop == "SAME_LOWER") { pr = (k - 1) / 2; pl = k - 1 - pr; }
        else if (autop == "NOTSET") {
            std::vector<int64_t> pads = n->attr_ints("pads") ? *n->attr_ints("pads") : std::vector<int64_t>(two_d ? 4 : 2, 0);
            if (two_d) { if (pads.size() != 4 || pads[0] || pads[2]) PLAN_FAIL("Conv '%s': pads", n->name.c_str()); pl = (int)pads[1]; pr = (int)pads[3]; }
            else { if (pads.size() != 2) PLAN_FAIL("Conv '%s': pads", n->name.c_str()); pl = (int)pads[0]; pr = (int)pads[1]; }
        } else PLAN_FAIL("Conv '%s': auto_pad %s", n->name.c_str(), autop.c_str());
        if (pl + pr != k - 1) PLAN_FAIL("Conv '%s': padding (%d, %d) does not keep the sequence length for width %d ('same' expected)", n->name.c_str(), pl, pr, k);
        ci.pl = pl;
        if (!W.to_f32(ci.W)) PLAN_FAIL("cannot decode Conv weights");
        ci.b.assign((size_t)ci.F, 0.f);
        if (!n->input(2).empty()) {
            auto b = ix.cst.find(n->input(2));
            if (b == ix.cst.end() || b->second->numel() != ci.F || !b->second->to_f32(ci.b)) PLAN_FAIL("Conv '%s': bias is not a constant [F] tensor", n->name.c_str());
        }
        ci.wname = n->input(1);
        info[n->out[0]] = ci;
    }
    auto only = [&](const std::vector<const Node *> &v) -> const Node * {
        std::set<const Node *> u(v.begin(), v.end());
        return u.size() == 1 ? *u.begin() : nullptr;
    };
    std::vector<std::string> order;
    std::string cur;
    if (convs.size() > 1) {
        std::vector<const Node *> nxt;
        for (auto *n : convs) ix.fwd(n->out[0], nxt);
        const Node *cat = only(nxt);
        if (!cat || cat->op != "Concat" || (cat->attr_i("axis", 0) != 1 && cat->attr_i("axis", 0) != -2))
            PLAN_FAIL("Conv outputs are not concatenated over the channel axis (axis 1 of [b, F, L])");
        for (auto &i : cat->in) order.push_back(ix.back(i));
        std::set<std::string> a(order.begin(), order.end());
        if (a.size() != info.size() || order.size() != info.size()) PLAN_FAIL("Concat inputs are not exactly the Conv outputs");
        for (auto &o : order) if (!info.count(o)) PLAN_FAIL("Concat inputs are not exactly the Conv outputs");
        cur = cat->out[0];
    } else { order = {convs[0]->out[0]}; cur = order[0]; }
    std::vector<float> bias;
    for (size_t l = 0; l < order.size(); ++l) {
        const ConvInfo &ci = info[order[l]];
        plan.conv_W.push_back(ci.W); plan.conv_filters.push_back(ci.F); plan.conv_width.push_back(ci.w); plan.conv_pad_left.push_back(ci.pl);
        bias.insert(bias.end(), ci.b.begin(), ci.b.end());
        plan.roles[fmt("conv%zu_W", l + 1)] = ci.wname;
    }
    const int tot = (int)bias.size();
    plan.scale.assign((size_t)tot, 1.f);
    plan.shift = bias;
    const Node *n = only(ix.fwd(cur));
    if (!n) PLAN_FAIL("expected exactly one consumer after the concatenation");
    if (n->op == "BatchNormalization") {
        std::vector<double> p[4];
        for (int k = 0; k < 4; ++k) {
            auto t = ix.cst.find(n->input((size_t)k + 1));
            if (t == ix.cst.end()) PLAN_FAIL("BatchNormalization parameters are not constant");
            if (!t->second->to_f64(p[k]) || (int)p[k].size() != tot) PLAN_FAIL("BatchNormalization width does not match the concatenated filters");
        }
        const double e = (double)n->attr_f("epsilon", 1e-5f);
        for (int c = 0; c < tot; ++c) {
            const double s = p[0][(size_t)c] / sqrt(p[3][(size_t)c] + e);
            plan.scale[(size_t)c] = (float)s;
            plan.shift[(size_t)c] = (float)(((double)bias[(size_t)c] - p[2][(size_t)c]) * s + p[1][(size_t)c]);
        }
        n = only(ix.fwd(n->out[0]));
        if (!n) PLAN_FAIL("expected exactly one consumer after BatchNormalization");
    }
    if (n->op != "Relu") PLAN_FAIL("expected ReLU before the pooling, found %s", n->op.c_str());
    n = only(ix.fwd(n->out[0]));
    if (!n) PLAN_FAIL("expected exactly one consumer after ReLU");
    if (n->op == "ReduceMax") {
        auto *ax = n->attr_ints("axes");
        std::vector<int64_t> axes = ax ? *ax : std::vector<int64_t>();
        if (!ax && !n->input(1).empty()) { auto t = ix.cst.find(n->input(1)); if (t != ix.cst.end()) { std::vector<double> d; t->second->to_f64(d); for (double x : d) axes.push_back((int64_t)x); } }
        if (axes != std::vector<int64_t>{2} && axes != std::vector<int64_t>{-1}) PLAN_FAIL("ReduceMax is not over the residue axis of [b, F, L]");
    } else if (n->op != "GlobalMaxPool") PLAN_FAIL("expected a global max-pool over residues, found %s", n->op.c_str());
    n = only(ix.fwd(n->out[0]));
    if (!n || (n->op != "MatMul" && n->op != "Gemm") || !ix.is_const(n->input(1)))
        PLAN_FAIL("expected the FuncPredictor dense layer after the max-pool, found %s", n ? n->op.c_str() : "several consumers");
    Dense d;
    d.node = n; d.wname = n->input(1);
    const Tensor *w = ix.cst.at(d.wname);
    std::vector<float> raw;
    if (w->dims.size() != 2 || !w->to_f32(raw)) PLAN_FAIL("output layer weight %s is not a matrix", dims_str(*w).c_str());
    d.rows = (int)w->dims[0]; d.cols = (int)w->dims[1]; d.W = raw;
    if (n->op == "Gemm") {
        if (n->attr_i("transA", 0) || n->attr_f("alpha", 1.f) != 1.f || n->attr_f("beta", 1.f) != 1.f) PLAN_FAIL("Gemm with transA / alpha / beta is not supported");
        if (n->attr_i("transB", 0)) { std::swap(d.rows, d.cols); for (int r = 0; r < d.rows; ++r) for (int c = 0; c < d.cols; ++c) d.W[(size_t)r * d.cols + c] = raw[(size_t)c * d.rows + r]; }
        if (!n->input(2).empty()) { auto b = ix.cst.find(n->input(2)); if (b == ix.cst.end() || !b->second->to_f32(d.bias)) PLAN_FAIL("Gemm bias is not constant"); }
    }
    if (d.rows != tot || d.cols % 2) PLAN_FAIL("output layer weight (%d, %d) does not follow %d pooled channels", d.rows, d.cols, tot);
    if (!dense_bias_after(ix, d)) PLAN_FAIL("cannot decode the output bias");
    if (!d.bias.empty() && (int)d.bias.size() != d.cols) PLAN_FAIL("output bias width mismatch");
    const Node *smx = only(ix.fwd(d.out));
    const int64_t ax = smx ? smx->attr_i("axis", -1) : 0;
    if (!smx || smx->op != "Softmax" || g.outputs.empty() || smx->out[0] != g.outputs[0].name || (ax != -1 && ax != 2))
        PLAN_FAIL("graph does not end in a Softmax over the last axis");
    plan.out_W = d.W; plan.out_b = d.bias; plan.C = d.cols / 2;
    plan.roles["out_W"] = d.wname;
    if (!d.bias_name.empty()) plan.roles["out_b"] = d.bias_name;
    return true;
}

// rc: MDF_OK, MDF_ENOENT (cannot open), MDF_EPARSE (not an ONNX protobuf), MDF_EUNSUPPORTED (graph not recognised)
static int load_plan(const char *path, Plan &plan)
{
    FILE *fh = fopen(path, "rb");
    if (!fh) { set_error("%s: cannot open model file: %s", path, strerror(errno)); return MDF_ENOENT; }
    std::vector<uint8_t> buf;
    uint8_t chunk[1 << 16];
    size_t got;
    while ((got = fread(chunk, 1, sizeof chunk, fh)) > 0) buf.insert(buf.end(), chunk, chunk + got);
    fclose(fh);
    Model m;
    if (buf.empty() || !parse_model(buf.data(), buf.size(), m)) { set_error("%s: cannot parse as ONNX protobuf", path); return MDF_EPARSE; }
    const bool ok = m.g.inputs.size() == 1 ? recognise_cnn(m, plan) : recognise_gcn(m, plan);
    if (!ok) { set_error("%s: %s", path, plan.error.c_str()); return MDF_EUNSUPPORTED; }
    return MDF_OK;
}

static void json_str(std::string &o, const std::string &s)
{
    o += '"';
    for (char c : s) { if (c == '"' || c == '\\') { o += '\\'; o += c; } else if ((unsigned char)c < 0x20) o += fmt("\\u%04x", c); else o += c; }
    o += '"';
}

}  // namespace onnx
}  // namespace mdf

using namespace mdf;
using namespace mdf::onnx;

static const float *ptr_or_null(const std::vector<float> &v) { return v.empty() ? nullptr : v.data(); }

extern "C" int mdf_onnx_inspect(const char *onnx_path, char *buf, size_t capacity)
{
    MDF_REQUIRE(onnx_path && buf && capacity > 0, "mdf_onnx_inspect: bad arguments");
    Plan p;
    MDF_TRY(load_plan(onnx_path, p));
    std::string o = "{\"kind\": ";
    o += p.is_cnn ? "\"cnn\"" : "\"gcn\"";
    o += ", \"input_names\": [";
    for (size_t i = 0; i < p.input_names.size(); ++i) { if (i) o += ", "; json_str(o, p.input_names[i]); }
    o += fmt("], \"n_terms\": %d", p.C);
    if (p.is_cnn) {
        auto list = [&](const char *k, const std::vector<int> &v) { o += fmt(", \"%s\": [", k); for (size_t i = 0; i < v.size(); ++i) o += (i ? ", " : "") + std::to_string(v[i]); o += "]"; };
        list("conv_filters", p.conv_filters); list("conv_width", p.conv_width); list("conv_pad_left", p.conv_pad_left);
        double cs = 0, ch = 0;
        for (float v : p.scale) cs += v;
        for (float v : p.shift) ch += v;
        o += fmt(", \"scale_sum\": %.9g, \"shift_sum\": %.9g", cs, ch);
    } else {
        o += fmt(", \"lstm_hidden\": %d, \"n_lstm\": %zu, \"lm_dim\": %d, \"fc_dim\": %d, \"gc_activation\": %d, \"gc_alpha\": %.9g, \"eps\": %.9g, \"gc_dims\": [",
                 p.H, p.lstm_W.size(), p.E, p.F, p.act, p.alpha, p.eps);
        for (size_t i = 0; i < p.gc_dims.size(); ++i) o += (i ? ", " : "") + std::to_string(p.gc_dims[i]);
        o += fmt("], \"lm_fingerprint\": \"%016llx\"", p.lm_hash);
    }
    o += ", \"roles\": {";
    bool first = true;
    for (auto &kv : p.roles) { if (!first) o += ", "; first = false; json_str(o, kv.first); o += ": "; json_str(o, kv.second); }
    o += "}}";
    MDF_REQUIRE(o.size() + 1 <= capacity, "mdf_onnx_inspect: buffer too small (%zu bytes needed)", o.size() + 1);
    memcpy(buf, o.c_str(), o.size() + 1);
    return MDF_OK;
}

// the recognised weight playing `role`, as the pipeline will use it (Gemm transposes undone, conv bias + BatchNormalization folded)
extern "C" int mdf_onnx_tensor(const char *onnx_path, const char *role, float *buf, int64_t capacity, int64_t *count)
{
    MDF_REQUIRE(onnx_path && role && count, "mdf_onnx_tensor: bad arguments");
    Plan p;
    MDF_TRY(load_plan(onnx_path, p));
    const std::string r = role;
    const std::vector<float> *v = nullptr;
    auto layer = [&](const char *prefix, const char *suffix, const std::vector<std::vector<float>> &set) {
        for (size_t l = 0; l < set.size(); ++l) if (r == fmt("%s%zu%s", prefix, l + 1, suffix)) v = &set[l];
    };
    if (r == "aa_W") v = &p.aa_W; else if (r == "lm_W") v = &p.lm_W; else if (r == "lm_b") v = &p.lm_b;
    else if (r == "fc_W") v = &p.fc_W; else if (r == "fc_b") v = &p.fc_b; else if (r == "out_W") v = &p.out_W; else if (r == "out_b") v = &p.out_b;
    else if (r == "scale") v = &p.scale; else if (r == "shift") v = &p.shift;
    layer("lstm", "_W", p.lstm_W); layer("lstm", "_R", p.lstm_R); layer("lstm", "_B", p.lstm_B);
    layer("gc", "_W", p.gc_W); layer("gc", "_b", p.gc_b); layer("conv", "_W", p.conv_W);
    MDF_REQUIRE(v != nullptr, "mdf_onnx_tensor: unknown role '%s'", role);
    *count = (int64_t)v->size();
    if (!buf) return MDF_OK;
    MDF_REQUIRE(capacity >= *count, "mdf_onnx_tensor: buffer too small (%lld < %lld)", (long long)capacity, (long long)*count);
    if (!v->empty()) memcpy(buf, v->data(), v->size() * sizeof(float));
    return MDF_OK;
}

extern "C" int mdf_model_load(mdf_ctx *ctx, const char *onnx_path, mdf_model **out)
{
    MDF_REQUIRE(ctx && onnx_path && out, "mdf_model_load: bad arguments");
    Plan p;
    MDF_TRY(load_plan(onnx_path, p));
    if (p.is_cnn) { set_error("%s: single-input model: this is a sequence-only DeepCNN head, use mdf_cnn_model_load", onnx_path); return MDF_EUNSUPPORTED; }
    if (p.lstm_W.size() > MDF_MAX_LSTM) {
        set_error("%s: %zu LSTM layers: the engines take at most %d", onnx_path, p.lstm_W.size(), MDF_MAX_LSTM);
        return MDF_EUNSUPPORTED;
    }
    if (p.gc_W.size() > MDF_MAX_GC) {
        set_error("%s: %zu GraphConv layers: the engines take at most %d", onnx_path, p.gc_W.size(), MDF_MAX_GC);
        return MDF_EUNSUPPORTED;
    }
    mdf_model_desc d;
    memset(&d, 0, sizeof d);
    d.n_channels = 26; d.lstm_hidden = p.H; d.n_lstm = (int)p.lstm_W.size();
    for (int l = 0; l < d.n_lstm; ++l) { d.lstm_W[l] = p.lstm_W[(size_t)l].data(); d.lstm_R[l] = p.lstm_R[(size_t)l].data(); d.lstm_B[l] = ptr_or_null(p.lstm_B[(size_t)l]); }
    d.lm_dim = p.E; d.aa_W = p.aa_W.data(); d.lm_W = p.lm_W.data(); d.lm_b = ptr_or_null(p.lm_b);
    d.n_gc = (int)p.gc_W.size();
    for (int l = 0; l < d.n_gc; ++l) { d.gc_dims[l] = p.gc_dims[(size_t)l]; d.gc_W[l] = p.gc_W[(size_t)l].data(); d.gc_b[l] = ptr_or_null(p.gc_b[(size_t)l]); }
    d.gc_activation = p.act; d.gc_alpha = p.alpha; d.eps = p.eps;
    d.fc_dim = p.F; d.fc_W = p.fc_W.data(); d.fc_b = ptr_or_null(p.fc_b);
    d.n_terms = p.C; d.out_W = p.out_W.data(); d.out_b = ptr_or_null(p.out_b);
    return mdf_model_create(ctx, &d, out);
}

extern "C" int mdf_cnn_model_load(mdf_ctx *ctx, const char *onnx_path, mdf_cnn_model **out)
{
    MDF_REQUIRE(ctx && onnx_path && out, "mdf_cnn_model_load: bad arguments");
    Plan p;
    MDF_TRY(load_plan(onnx_path, p));
    if (!p.is_cnn) { set_error("%s: two-input model: this is a GCN head, use mdf_model_load", onnx_path); return MDF_EUNSUPPORTED; }
    if (p.conv_W.size() > MDF_MAX_CONV) {
        set_error("%s: DeepCNN model has %zu parallel Conv layers: the kernel takes at most %d", onnx_path, p.conv_W.size(), MDF_MAX_CONV);
        return MDF_EUNSUPPORTED;
    }
    mdf_cnn_desc d;
    memset(&d, 0, sizeof d);
    d.n_channels = 26; d.n_conv = (int)p.conv_W.size();
    for (int l = 0; l < d.n_conv; ++l) {
        d.conv_width[l] = p.conv_width[(size_t)l]; d.conv_filters[l] = p.conv_filters[(size_t)l]; d.conv_pad_left[l] = p.conv_pad_left[(size_t)l];
        d.conv_W[l] = p.conv_W[(size_t)l].data();
    }
    d.scale = p.scale.data(); d.shift = p.shift.data();
    d.n_terms = p.C; d.out_W = p.out_W.data(); d.out_b = ptr_or_null(p.out_b);
    return mdf_cnn_model_create(ctx, &d, out);
}

extern "C" int mdf_model_info(const mdf_model *m, int *n_terms, int *lstm_hidden, int *lm_dim, int *n_gc, int *gc_dims, int *fc_dim)
{
    MDF_REQUIRE(m, "mdf_model_info: model is NULL");
    if (n_terms) *n_terms = m->C;
    if (lstm_hidden) *lstm_hidden = m->H;
    if (lm_dim) *lm_dim = m->E;
    if (n_gc) *n_gc = m->n_gc;
    if (gc_dims) for (int l = 0; l < m->n_gc; ++l) gc_dims[l] = m->gc[l];
    if (fc_dim) *fc_dim = m->F;
    return MDF_OK;
}
