// host_module.cpp — CPython extension `loco_hd.loco_hd` (the reference's module path and name): the five classes of
// the reference's PyO3 boundary (/root/reference/src/lib.rs:9-17) written from scratch in C++/pybind11 because no
// Rust toolchain exists in this image.  It only validates, interns strings and marshals arrays; every `from_*`
// scoring call goes to CUDA through the C ABI (include/locohd_b200.h).  There is no CPU scoring path.
//
//   WeightFunction        weight_function.rs:5-121  (integral_* are host utilities, not on the hot path)
//   PrimitiveAtom         primitive_atom.rs:4-25
//   TagPairingRule        tag_pairing_rule.rs:5-77
//   StatisticalDistance   pmf/statistical_distances.rs:80-143
//   LoCoHD                locohd.rs:42-55, 286-568
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <limits>
#include <map>
#include <memory>
#include <mutex>
#include <optional>
#include <set>
#include <sstream>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "locohd_b200.h"

namespace py = pybind11;

namespace {

int g_device = -1;  // -1: LOCOHD_DEVICE or 0

int default_device() {
    if (g_device >= 0) return g_device;
    if (const char* e = std::getenv("LOCOHD_DEVICE")) return std::atoi(e);
    return 0;
}

[[noreturn]] void raise_status(int st, const char* msg) {
    std::string m = msg ? msg : "";
    if (st >= LOCOHD_ERR_CUDA) throw std::runtime_error(m);
    throw py::value_error(m);
}

// ------------------------------------------------------------------------------------------ WeightFunction
struct WeightFunction {
    std::string function_name;
    std::vector<double> parameters;
    int kind = 0;

    WeightFunction(std::string name, std::vector<double> params) : function_name(std::move(name)), parameters(std::move(params)) {
        const auto& p = parameters;
        auto need = [&](size_t n) {
            if (p.size() != n)
                throw py::value_error("For function \"" + function_name + "\" there must be exactly " + std::to_string(n) + " parameters!");
        };
        if (function_name == "hyper_exp") {  // weight_function.rs:31-40
            kind = LOCOHD_WF_HYPER_EXP;
            if (p.size() % 2 != 0) throw py::value_error("For function \"hyper_exp\" there must be an even number of parameters!");
            for (double v : p)
                if (v <= 0.0) throw py::value_error("For function \"hyper_exp\" all parameters must be positive!");
        } else if (function_name == "dagum") {  // :42-50
            kind = LOCOHD_WF_DAGUM;
            need(3);
            if (p[0] < 0.0 || p[1] < 0.0 || p[2] < 0.0) throw py::value_error("For function \"dagum\" all parameters must be positive!");
        } else if (function_name == "uniform") {  // :53-67
            kind = LOCOHD_WF_UNIFORM;
            need(2);
            if (p[0] < 0.0) throw py::value_error("For function \"uniform\" the first parameter must be non-negative!");
            if (p[1] <= 0.0) throw py::value_error("For function \"uniform\" the second parameter must be positive!");
            if (p[0] >= p[1]) throw py::value_error("For function \"uniform\" the first parameter must be smaller than the second!");
        } else if (function_name == "kumaraswamy") {  // :69-83
            kind = LOCOHD_WF_KUMARASWAMY;
            need(4);
            if (p[0] < 0.0) throw py::value_error("For function \"kumaraswamy\" the first parameter must be non-negative!");
            if (p[1] <= 0.0 || p[2] <= 0.0 || p[3] <= 0.0)
                throw py::value_error("For function \"kumaraswamy\" after the first parameter all parameters must be positive!");
            if (p[0] >= p[1]) throw py::value_error("For function \"kumaraswamy\" the first parameter must be smaller than the second!");
        } else {
            throw py::value_error("No function implemented with name \"" + function_name + "\"!");
        }
        if (p.size() > LOCOHD_MAX_WF_PARAMS)
            throw py::value_error("at most " + std::to_string(LOCOHD_MAX_WF_PARAMS) + " weight function parameters are supported");
    }

    double cdf(double x) const {  // cdfs.rs:5-63
        const auto& p = parameters;
        switch (kind) {
            case LOCOHD_WF_HYPER_EXP: {
                double norm = 0.0, sum = 0.0;
                const size_t h = p.size() / 2;
                for (size_t i = 0; i < h; ++i) { sum += p[i] * std::exp(-p[h + i] * x); norm += p[i]; }
                return 1.0 - sum / norm;
            }
            case LOCOHD_WF_DAGUM: return std::pow(1.0 + std::pow(x / p[1], -p[0]), -p[2]);
            case LOCOHD_WF_UNIFORM:
                if (x < p[0]) return 0.0;
                if (x > p[1]) return 1.0;
                return (x - p[0]) / (p[1] - p[0]);
            default: {
                if (x < p[0]) return 0.0;
                if (x > p[1]) return 1.0;
                const double z = (x - p[0]) / (p[1] - p[0]);
                return 1.0 - std::pow(1.0 - std::pow(z, p[2]), p[3]);
            }
        }
    }
    double integral_point(double x) const {  // weight_function.rs:95-103
        if (x < 0.0) {
            std::ostringstream os;
            os << "Invalid input value: " << x << ". All values must be non-negative!";
            throw py::value_error(os.str());
        }
        return cdf(x);
    }
    std::vector<double> integral_vec(const std::vector<double>& xs) const {
        std::vector<double> out;
        out.reserve(xs.size());
        for (double x : xs) out.push_back(integral_point(x));
        return out;
    }
    double integral_range(double from, double to) const { return integral_point(to) - integral_point(from); }

    locohd_weight_function abi() const {
        locohd_weight_function w{};
        w.kind = kind;
        w.n_params = (int32_t)parameters.size();
        for (size_t i = 0; i < parameters.size(); ++i) w.params[i] = parameters[i];
        return w;
    }
};

// ------------------------------------------------------------------------------------------- PrimitiveAtom
struct PrimitiveAtom {
    std::string primitive_type;
    std::string tag;
    std::array<double, 3> coordinates;
};

// ------------------------------------------------------------------------------------------ TagPairingRule
struct TagPairingRule {
    bool with_list = false;
    bool accept_same = true;
    std::set<std::pair<std::string, std::string>> tag_pairs;
    bool accepted_pairs = true;
    bool ordered = true;

    static bool as_bool(const py::handle& h, bool* out) {
        if (py::isinstance<py::bool_>(h)) { *out = h.cast<bool>(); return true; }
        // numpy.bool_
        if (std::string(py::str(py::type::of(h).attr("__name__"))).rfind("bool", 0) == 0) { *out = py::bool_(h.attr("__bool__")()); return true; }
        return false;
    }

    explicit TagPairingRule(const py::dict& variant) {
        // the enum tries WithoutList first, then WithList (tag_pairing_rule.rs:5-21)
        if (variant.contains("accept_same") && as_bool(variant["accept_same"], &accept_same)) {
            with_list = false;
            return;
        }
        bool ok = variant.contains("tag_pairs") && variant.contains("accepted_pairs") && variant.contains("ordered");
        if (ok) ok = as_bool(variant["accepted_pairs"], &accepted_pairs) && as_bool(variant["ordered"], &ordered);
        if (ok) {
            try {
                for (auto item : variant["tag_pairs"]) {
                    auto t = item.cast<py::tuple>();
                    if (t.size() != 2) throw py::type_error("");
                    tag_pairs.emplace(t[0].cast<std::string>(), t[1].cast<std::string>());
                }
            } catch (const std::exception&) {
                ok = false;
            }
        }
        if (!ok)
            throw py::type_error(
                "failed to extract enum TagPairingRuleVariants ('WithoutList | WithList'): expected a dict with the key "
                "'accept_same' (bool) or with the keys 'tag_pairs' (set of 2-tuples of str), 'accepted_pairs' (bool) and 'ordered' (bool)");
        with_list = true;
    }
    TagPairingRule() = default;

    bool pair_accepted(const std::pair<std::string, std::string>& pair) const {  // tag_pairing_rule.rs:49-76
        if (!with_list) {
            bool acc = pair.first == pair.second;
            if (!accept_same) acc = !acc;
            return acc;
        }
        bool acc = tag_pairs.count(pair) > 0;
        if (!ordered) acc = acc || tag_pairs.count({pair.second, pair.first}) > 0;
        if (!accepted_pairs) acc = !acc;
        return acc;
    }

    std::string dbg() const {  // `{:#?}` of the Rust struct (tag_pairing_rule.rs:42-44)
        std::ostringstream os;
        os << "TagPairingRule {\n    variant: ";
        if (!with_list) {
            os << "WithoutList {\n        accept_same: " << (accept_same ? "true" : "false") << ",\n    },\n}";
        } else {
            os << "WithList {\n        tag_pairs: {\n";
            for (const auto& p : tag_pairs) os << "            (\n                \"" << p.first << "\",\n                \"" << p.second << "\",\n            ),\n";
            os << "        },\n        accepted_pairs: " << (accepted_pairs ? "true" : "false") << ",\n        ordered: "
               << (ordered ? "true" : "false") << ",\n    },\n}";
        }
        return os.str();
    }
};

// ------------------------------------------------------------------------------------- StatisticalDistance
struct StatisticalDistance {
    std::string name;
    std::vector<double> parameters;
    int kind = 0;

    StatisticalDistance(std::string n, std::vector<double> p) : name(std::move(n)), parameters(std::move(p)) {
        size_t want;  // statistical_distances.rs:106-119
        if (name == "Hellinger") { kind = LOCOHD_SD_HELLINGER; want = 1; }
        else if (name == "Kolmogorov-Smirnov") { kind = LOCOHD_SD_KOLMOGOROV_SMIRNOV; want = 0; }
        else if (name == "Kullback-Leibler") { kind = LOCOHD_SD_KULLBACK_LEIBLER; want = 1; }
        else if (name == "Renyi") { kind = LOCOHD_SD_RENYI; want = 2; }
        else throw py::value_error("Invalid statistical distance name " + name + "!");
        if (parameters.size() != want)
            throw py::value_error("Invalid number of parameters for " + name + ": " + std::to_string(parameters.size()));
    }

    static double kl(const std::vector<double>& a, const std::vector<double>& b, double eps) {
        double d = 0.0;
        for (size_t i = 0; i < std::min(a.size(), b.size()); ++i) d += a[i] * std::log((a[i] + eps) / (b[i] + eps));
        return d;
    }
    double run(const std::vector<double>& a, const std::vector<double>& b) const {  // statistical_distances.rs:4-142
        const size_t n = std::min(a.size(), b.size());
        switch (kind) {
            case LOCOHD_SD_HELLINGER: {
                const double e = parameters[0];
                double d = 0.0;
                for (size_t i = 0; i < n; ++i) d += std::pow(std::fabs(std::pow(a[i], 1.0 / e) - std::pow(b[i], 1.0 / e)), e);
                return std::pow(d / 2.0, 1.0 / e);
            }
            case LOCOHD_SD_KOLMOGOROV_SMIRNOV: {
                if (n == 0) throw py::value_error("empty distributions");
                double best = 0.0;
                for (size_t i = 0; i < n; ++i) best = std::max(best, std::fabs(a[i] - b[i]));
                return best;
            }
            case LOCOHD_SD_KULLBACK_LEIBLER: return kl(a, b, parameters[0]);
            default: {
                const double alpha = parameters[0], eps = parameters[1];
                if (alpha == 1.0) return kl(a, b, eps);
                if (std::isinf(alpha) && alpha > 0) {
                    if (n == 0) throw py::value_error("empty distributions");
                    double best = (a[0] + eps) / (b[0] + eps);
                    for (size_t i = 1; i < n; ++i) best = std::max(best, (a[i] + eps) / (b[i] + eps));
                    return std::log(best);
                }
                if (alpha == 0.0) {
                    double s = 0.0;
                    for (size_t i = 0; i < n; ++i) if (a[i] > 0.0) s += b[i];
                    return -std::log(s);
                }
                double s = 0.0;
                for (size_t i = 0; i < n; ++i) s += a[i] * std::pow((a[i] + eps) / (b[i] + eps), alpha - 1.0);
                return std::log(s) / (alpha - 1.0);
            }
        }
    }
};

// -------------------------------------------------------------------------------------------------- LoCoHD
// One CUDA context and the mutex that serialises the C-ABI calls on it (a context owns one stream).  Locking
// discipline: the mutex is only ever taken with the GIL RELEASED and is dropped before the GIL comes back, so a
// thread never waits for one while holding the other (two Python threads may share a LoCoHD instance, as they can
// upstream, where the GIL simply serialises them).  Python-side state (tag table, context pointer) is only touched
// with the GIL held.
struct Dev {
    locohd_ctx* c = nullptr;
    int device = -1;
    std::mutex mu;
    ~Dev() { if (c) locohd_ctx_destroy(c); }
};

// Runs f(ctx) -> status without the GIL and under the device mutex; raises with the context's message.
template <class F>
void device_call(const std::shared_ptr<Dev>& d, F&& f) {
    int st;
    std::string msg;
    {
        py::gil_scoped_release rel;
        std::lock_guard<std::mutex> g(d->mu);
        st = f(d->c);
        if (st) msg = locohd_last_error(d->c);
    }   // the mutex is released first, then the GIL is taken again
    if (st) raise_status(st, msg.c_str());
}

using F64Array = py::array_t<double, py::array::c_style | py::array::forcecast>;
using U16Array = py::array_t<uint16_t, py::array::c_style | py::array::forcecast>;
using U32Array = py::array_t<uint32_t, py::array::c_style | py::array::forcecast>;
using U64Array = py::array_t<uint64_t, py::array::c_style | py::array::forcecast>;

// Device-resident structures / environments handed out by LoCoHD.structures / LoCoHD.environments (SURVEY 8(f) N1).
// They keep the context alive; destruction only enqueues stream-ordered frees and needs no lock.
struct Structures {
    std::shared_ptr<Dev> dev;
    locohd_structs* h = nullptr;
    uint64_t n_structs = 0, n_prims = 0;
    std::vector<uint64_t> offsets;
    ~Structures() { close(); }
    void close() { if (h) { locohd_structs_destroy(h); h = nullptr; } }
    void need() const { if (!h) throw py::value_error("structures have been closed"); }
    void update_xyz(const py::array& xyz) {
        need();
        if ((uint64_t)xyz.size() != 3 * n_prims) throw py::value_error("xyz must hold 3 coordinates per primitive of the set");
        if (py::isinstance<py::array_t<float>>(xyz)) {   // float32 goes over the f32 wire (exact widening on the device)
            auto a = py::array_t<float, py::array::c_style | py::array::forcecast>::ensure(xyz);
            device_call(dev, [&](locohd_ctx*) { return locohd_structs_update_xyz_f32(h, a.data()); });
        } else {
            auto a = F64Array::ensure(xyz);
            if (!a) throw py::type_error("xyz must be a float array");
            device_call(dev, [&](locohd_ctx*) { return locohd_structs_update_xyz(h, a.data()); });
        }
    }
    // Frames of one compiled topology (PrimitiveAssigner.compile_topology): atoms -> centroids on the device.
    void update_from_atoms(const py::array_t<float, py::array::c_style | py::array::forcecast>& atoms,
                           const U32Array& segment_start, const U32Array& atom_index, uint64_t first_struct) {
        need();
        if (segment_start.size() < 1) throw py::value_error("segment_start must have n_primitives + 1 entries");
        if (atoms.ndim() < 2 || atoms.shape(atoms.ndim() - 1) != 3) throw py::value_error("atom coordinates must be [n_frames, n_atoms, 3] or [n_atoms, 3]");
        const uint64_t n_frames = atoms.ndim() == 3 ? (uint64_t)atoms.shape(0) : 1;
        const uint64_t n_atoms = (uint64_t)atoms.shape(atoms.ndim() - 2);
        const uint64_t n_prims_t = (uint64_t)segment_start.size() - 1;
        device_call(dev, [&](locohd_ctx*) {
            return locohd_structs_update_from_atoms(h, first_struct, n_frames, n_atoms, atoms.data(), n_prims_t,
                                                    segment_start.data(), atom_index.data(), (uint64_t)atom_index.size());
        });
    }
};

struct Environments {
    std::shared_ptr<Dev> dev;
    locohd_envset* h = nullptr;
    uint64_t n_env = 0;
    ~Environments() { close(); }
    void close() { if (h) { locohd_envset_destroy(h); h = nullptr; } }
};

std::vector<std::string> to_strings(const py::handle& seq, const char* what) {
    if (py::isinstance<py::str>(seq)) throw py::type_error(std::string(what) + ": can't extract `str` to a list");
    std::vector<std::string> out;
    for (auto item : seq) out.push_back(item.cast<std::string>());
    return out;
}

struct LoCoHD {
    std::vector<std::string> category_names;
    std::unordered_map<std::string, uint16_t> category_index;
    std::vector<double> category_weights;
    bool multiple_wf = false;
    std::vector<std::string> wf_keys;          // Multiple: sorted keys; Single: {""}
    std::vector<WeightFunction> wfs;
    std::unordered_map<std::string, uint32_t> wf_index;
    TagPairingRule rule;
    StatisticalDistance sd{"Hellinger", {2.0}};
    // device side, created at the first scoring call (GIL held whenever these are touched)
    std::shared_ptr<Dev> dev;
    std::unordered_map<std::string, uint32_t> tag_ids;   // grows with every new tag seen

    LoCoHD(const py::object& categories, const py::object& w_func, const py::object& tag_pairing_rule,
           const py::object& n_of_threads, const py::object& weights, const py::object& statistical_distance) {
        category_names = to_strings(categories, "categories");
        if (category_names.empty())  // locohd.rs:305-309
            throw py::value_error("The number of possible categories (primitive types) cannot be zero!");
        for (size_t i = 0; i < category_names.size(); ++i) {
            if (!category_index.emplace(category_names[i], (uint16_t)i).second)
                throw py::value_error("Duplicate category name \"" + category_names[i] + "\"!");
        }
        if (category_names.size() > LOCOHD_MAX_CATEGORIES)
            throw py::value_error("At most " + std::to_string(LOCOHD_MAX_CATEGORIES) + " categories are supported by the CUDA path!");
        if (weights.is_none()) category_weights.assign(category_names.size(), 1.0);
        else category_weights = weights.cast<std::vector<double>>();
        if (category_weights.size() != category_names.size())  // locohd.rs:325-333
            throw py::value_error("LoCoHD parameters 'categories' and 'category_weights' must have the same lengths! Instead, they have lengths of " +
                                  std::to_string(category_names.size()) + " vs. " + std::to_string(category_weights.size()) + "!");
        size_t bad = 0;
        for (double w : category_weights) if (w <= 0.0 || std::isnan(w)) ++bad;
        if (bad)  // locohd.rs:335-346
            throw py::value_error("LoCoHD parameter 'category_weights' must only contain positive values! Instead, it contains " +
                                  std::to_string(bad) + " non-positive values!");
        if (w_func.is_none()) {  // locohd.rs:349-354
            wfs.emplace_back("uniform", std::vector<double>{3.0, 10.0});
            wf_keys = {""};
        } else if (py::isinstance<WeightFunction>(w_func)) {
            wfs.push_back(w_func.cast<WeightFunction>());
            wf_keys = {""};
        } else if (py::isinstance<py::dict>(w_func)) {
            multiple_wf = true;
            std::map<std::string, WeightFunction> sorted;
            for (auto kv : w_func.cast<py::dict>()) {
                if (!py::isinstance<py::str>(kv.first) || !py::isinstance<WeightFunction>(kv.second))
                    throw py::type_error("w_func must be a WeightFunction or a dict[str, WeightFunction]");
                sorted.emplace(kv.first.cast<std::string>(), kv.second.cast<WeightFunction>());
            }
            for (auto& kv : sorted) {
                wf_index.emplace(kv.first, (uint32_t)wfs.size());
                wf_keys.push_back(kv.first);
                wfs.push_back(kv.second);
            }
        } else {
            throw py::type_error("w_func must be a WeightFunction or a dict[str, WeightFunction]");
        }
        if (!tag_pairing_rule.is_none()) rule = tag_pairing_rule.cast<TagPairingRule>();  // default accept_same=true, locohd.rs:357-362
        if (!statistical_distance.is_none()) sd = statistical_distance.cast<StatisticalDistance>();
        if (!n_of_threads.is_none()) {
            // accepted for signature compatibility (rayon pool size upstream, locohd.rs:372-383); the GPU grid replaces it
            (void)n_of_threads.cast<size_t>();
        }
    }

    py::dict categories_dict() const {
        py::dict d;
        for (size_t i = 0; i < category_names.size(); ++i) d[py::str(category_names[i])] = i;
        return d;
    }
    py::object w_func_object() const {
        if (!multiple_wf) return py::cast(wfs[0]);
        py::dict d;
        for (size_t i = 0; i < wfs.size(); ++i) d[py::str(wf_keys[i])] = py::cast(wfs[i]);
        return d;
    }

    uint32_t intern_tag(const std::string& t) {
        auto it = tag_ids.find(t);
        if (it != tag_ids.end()) return it->second;
        const uint32_t id = (uint32_t)tag_ids.size();
        tag_ids.emplace(t, id);
        return id;
    }
    uint16_t cat_id(const std::string& c) const {
        if (category_names.size() <= 16) {   // a handful of short names: a linear scan beats hashing the string
            for (size_t i = 0; i < category_names.size(); ++i)
                if (category_names[i] == c) return (uint16_t)i;
            return (uint16_t)LOCOHD_UNKNOWN_CATEGORY;
        }
        auto it = category_index.find(c);
        return it == category_index.end() ? (uint16_t)LOCOHD_UNKNOWN_CATEGORY : it->second;
    }

    // Creates the context on first use (or when the selected device changed) and sends the parameters.  Called
    // with the GIL held; a context still in use by another thread's call stays alive through its shared_ptr.
    std::shared_ptr<Dev> ensure_ctx() {
        const int want = default_device();
        if (dev && dev->device == want) return dev;
        locohd_ctx* c = nullptr;
        const int st = locohd_ctx_create(want, &c);
        if (st) raise_status(LOCOHD_ERR_CUDA, locohd_last_error(nullptr));
        auto fresh = std::make_shared<Dev>();
        fresh->c = c;
        fresh->device = want;
        std::vector<uint64_t> pairs;
        if (rule.with_list)
            for (const auto& p : rule.tag_pairs) pairs.push_back(((uint64_t)intern_tag(p.first) << 32) | intern_tag(p.second));
        std::vector<locohd_weight_function> w;
        for (const auto& f : wfs) w.push_back(f.abi());
        locohd_params p{};
        p.n_categories = (int32_t)category_names.size();
        p.category_weights = category_weights.data();
        p.sd_kind = sd.kind;
        p.sd_params[0] = sd.parameters.size() > 0 ? sd.parameters[0] : 0.0;
        p.sd_params[1] = sd.parameters.size() > 1 ? sd.parameters[1] : 0.0;
        p.n_weight_functions = (int32_t)w.size();
        p.weight_functions = w.data();
        p.tpr_kind = rule.with_list ? LOCOHD_TPR_WITH_LIST : LOCOHD_TPR_WITHOUT_LIST;
        p.tpr_accept_same = rule.accept_same;
        p.tpr_accepted_pairs = rule.accepted_pairs;
        p.tpr_ordered = rule.ordered;
        p.n_tag_pairs = pairs.size();
        p.tag_pairs = pairs.data();
        if (locohd_ctx_set_params(c, &p)) raise_status(LOCOHD_ERR_BAD_PARAM, locohd_last_error(c));   // not shared yet: no lock
        dev = fresh;
        return dev;
    }

    // keys_to_weight_functions (locohd.rs:230-283): returns per-anchor indices (empty = weight function 0 for all)
    std::vector<uint32_t> resolve_keys(const std::optional<std::vector<std::string>>& keys, size_t target_len) const {
        if (multiple_wf && keys) {
            if (keys->size() != target_len)
                throw py::value_error("The w_func_keys vector has an invalid length (" + std::to_string(keys->size()) +
                                      " instead of " + std::to_string(target_len) + ")!");
            std::vector<uint32_t> out;
            out.reserve(keys->size());
            size_t failed = 0;
            for (const auto& k : *keys) {
                auto it = wf_index.find(k);
                if (it == wf_index.end()) { ++failed; out.push_back(0); } else out.push_back(it->second);
            }
            if (failed)
                throw py::value_error("The vector contains " + std::to_string(failed) + " out of " + std::to_string(keys->size()) +
                                      " invalid weight function keys!");
            return out;
        }
        if (!multiple_wf && !keys) return {};
        throw py::value_error("Invalid pairing for the LoCoHD instance's w_func option and the method's w_func_keys parameter!");
    }

    std::vector<uint16_t> cat_ids(const std::vector<std::string>& seq) const {
        std::vector<uint16_t> out(seq.size());
        for (size_t i = 0; i < seq.size(); ++i) out[i] = cat_id(seq[i]);
        return out;
    }

    // ---- from_anchors (locohd.rs:392-406)
    double from_anchors(const py::object& seq_a, const py::object& seq_b, const std::vector<double>& da,
                        const std::vector<double>& db, const std::optional<std::string>& key) {
        const auto sa = cat_ids(to_strings(seq_a, "seq_a")), sb = cat_ids(to_strings(seq_b, "seq_b"));
        std::optional<std::vector<std::string>> keys;
        if (key) keys = std::vector<std::string>{*key};
        const auto idx = resolve_keys(keys, 1);
        const auto d = ensure_ctx();
        double out = 0.0;
        device_call(d, [&](locohd_ctx* c) {
            return locohd_score_anchor_lists(c, sa.data(), sa.size(), da.data(), da.size(), sb.data(), sb.size(),
                                             db.data(), db.size(), idx.empty() ? 0u : idx[0], &out);
        });
        return out;
    }

    // Two row sets (from_dmxs / from_coords) -> environments -> one job; everything inside one locked region.
    template <class Build>
    std::vector<double> score_rows(const std::shared_ptr<Dev>& d, size_t n, const std::vector<uint32_t>& wf, Build&& build) {
        std::vector<double> out(n);
        device_call(d, [&](locohd_ctx* c) {
            locohd_envset *ea = nullptr, *eb = nullptr;
            int st = build(c, &ea, &eb);
            if (!st) {
                const locohd_job job{0, 0, n};
                st = locohd_score_jobs(c, ea, eb, 1, &job, wf.empty() ? nullptr : wf.data(), out.data(), nullptr);
            }
            locohd_envset_destroy(ea);
            locohd_envset_destroy(eb);
            return st;
        });
        return out;
    }

    // ---- from_dmxs (locohd.rs:410-458)
    // A distance matrix as the reference takes it (Vec<Vec<f64>>): rows may have different lengths.
    struct Rows {
        std::vector<uint64_t> off{0};
        std::vector<double> val;
        size_t cols = 0;      // row length of rectangular input (a 2-D array or equally long nested lists)
        bool rect = false;
        size_t n() const { return off.size() - 1; }
        size_t max_len() const {
            size_t m = 0;
            for (size_t r = 0; r + 1 < off.size(); ++r) m = std::max<size_t>(m, off[r + 1] - off[r]);
            return m;
        }
    };
    static Rows to_rows(const py::object& m, const char* what) {
        Rows rows;
        auto a = F64Array::ensure(m);   // rectangular input (nested lists or an ndarray): one conversion
        if (a && a.ndim() == 2) {
            const size_t nr = a.shape(0), nc = a.shape(1);
            rows.val.assign(a.data(), a.data() + nr * nc);
            for (size_t r = 0; r < nr; ++r) rows.off.push_back((r + 1) * nc);
            rows.rect = true;
            rows.cols = nc;
            return rows;
        }
        PyErr_Clear();
        if (a && a.ndim() == 1 && a.shape(0) == 0) return rows;
        if (py::isinstance<py::str>(m)) throw py::type_error(std::string(what) + ": can't extract `str` to a list");
        try {
            for (auto row : m) {
                const auto v = row.cast<std::vector<double>>();
                rows.val.insert(rows.val.end(), v.begin(), v.end());
                rows.off.push_back(rows.val.size());
            }
        } catch (const py::cast_error&) {
            throw py::type_error(std::string(what) + " must be a sequence of sequences of floats");
        }
        return rows;
    }

    // The arguments of from_dmxs / from_dmxs_grad, converted and checked as the reference does.
    struct DmxCall {
        std::vector<uint16_t> sa, sb;
        Rows ma, mb;
        std::vector<uint32_t> wf;
        size_t n_rows() const { return ma.n(); }
    };
    DmxCall dmx_call(const py::object& seq_a, const py::object& seq_b, const py::object& dmx_a, const py::object& dmx_b,
                     const std::optional<std::vector<std::string>>& keys) const {
        DmxCall a;
        a.sa = cat_ids(to_strings(seq_a, "seq_a"));
        a.sb = cat_ids(to_strings(seq_b, "seq_b"));
        a.ma = to_rows(dmx_a, "dmx_a");
        a.mb = to_rows(dmx_b, "dmx_b");
        const size_t rows_a = a.ma.n(), rows_b = a.mb.n();
        if (rows_a != rows_b)  // locohd.rs:420-428
            throw py::value_error("Expected matrices with the same length, got lengths " + std::to_string(rows_a) + " and " +
                                  std::to_string(rows_b) + "!");
        a.wf = resolve_keys(keys, rows_a);
        if (rows_a == 0) return a;
        // sort_together indexes seq by the row's indices (utils.rs:33-36): a short seq panics upstream, a long one is cut
        if (a.sa.size() < a.ma.max_len() || a.sb.size() < a.mb.max_len())
            throw py::value_error("The category sequences are shorter than the distance matrix rows!");
        for (const Rows* m : {&a.ma, &a.mb})
            for (size_t r = 0; r < m->n(); ++r)
                if (m->off[r + 1] == m->off[r]) throw py::value_error("Empty distance matrix rows!");
        return a;
    }

    std::vector<double> from_dmxs(const py::object& seq_a, const py::object& seq_b, const py::object& dmx_a,
                                  const py::object& dmx_b, const std::optional<std::vector<std::string>>& keys) {
        const DmxCall a = dmx_call(seq_a, seq_b, dmx_a, dmx_b, keys);
        if (a.n_rows() == 0) return {};
        const auto d = ensure_ctx();
        auto build = [&](locohd_ctx* c, const Rows& m, const std::vector<uint16_t>& cats, locohd_envset** e) {
            return locohd_envset_from_ragged_rows(c, m.n(), m.off.data(), m.val.data(), cats.data(), cats.size(), e);
        };
        return score_rows(d, a.n_rows(), a.wf, [&](locohd_ctx* c, locohd_envset** ea, locohd_envset** eb) {
            int st = build(c, a.ma, a.sa, ea);
            if (!st) st = build(c, a.mb, a.sb, eb);
            return st;
        });
    }

    static const double* weights_of(const py::object& pair_weights, size_t n, F64Array& keep) {
        if (pair_weights.is_none()) return nullptr;
        keep = pair_weights.cast<F64Array>();
        if ((size_t)keep.size() != n) throw py::value_error("pair_weights must have one entry per row");
        return keep.data();
    }

    // from_dmxs with the gradients of the scores with respect to every matrix entry: (scores, grad_dmx_a, grad_dmx_b),
    // grad = pair_weights[r] dS_r / d dmx[r][c] (pair_weights None: all 1); [n_rows, row_len] arrays for rectangular
    // input, lists of 1-D arrays for ragged rows
    py::tuple from_dmxs_grad(const py::object& seq_a, const py::object& seq_b, const py::object& dmx_a,
                             const py::object& dmx_b, const std::optional<std::vector<std::string>>& keys,
                             const py::object& pair_weights) {
        const DmxCall a = dmx_call(seq_a, seq_b, dmx_a, dmx_b, keys);
        const size_t n = a.n_rows();
        F64Array pw;
        const double* w = weights_of(pair_weights, n, pw);
        py::array_t<double> out(n);
        std::vector<double> ga(a.ma.val.size()), gb(a.mb.val.size());
        if (n) {
            const auto d = ensure_ctx();
            double* o = out.mutable_data();
            device_call(d, [&](locohd_ctx* c) {
                return locohd_from_rows_grad(c, n, a.ma.off.data(), a.ma.val.data(), a.sa.data(), a.sa.size(),
                                             a.mb.off.data(), a.mb.val.data(), a.sb.data(), a.sb.size(),
                                             a.wf.empty() ? nullptr : a.wf.data(), w, o, ga.data(), gb.data());
            });
        }
        auto shape = [](const Rows& m, const std::vector<double>& g) -> py::object {
            if (m.rect) {
                py::array_t<double> r({(py::ssize_t)m.n(), (py::ssize_t)m.cols});
                std::copy(g.begin(), g.end(), r.mutable_data());
                return r;
            }
            py::list l;
            for (size_t r = 0; r < m.n(); ++r) {
                py::array_t<double> row((py::ssize_t)(m.off[r + 1] - m.off[r]));
                std::copy(g.begin() + m.off[r], g.begin() + m.off[r + 1], row.mutable_data());
                l.append(row);
            }
            return l;
        };
        return py::make_tuple(out, shape(a.ma, ga), shape(a.mb, gb));
    }

    // ---- from_coords (locohd.rs:463-476)
    // The arguments of from_coords / from_coords_grad, converted and checked as the reference does.
    struct CoordsCall {
        std::vector<uint16_t> sa, sb;
        F64Array xa, xb;
        size_t n = 0;
        std::vector<uint32_t> wf;
    };
    CoordsCall coords_call(const py::object& seq_a, const py::object& seq_b, const py::object& coords_a,
                           const py::object& coords_b, const std::optional<std::vector<std::string>>& keys) const {
        CoordsCall a;
        a.sa = cat_ids(to_strings(seq_a, "seq_a"));
        a.sb = cat_ids(to_strings(seq_b, "seq_b"));
        auto to_xyz = [](const py::object& m, const char* what) {
            auto a = F64Array::ensure(m);
            if (!a) { PyErr_Clear(); throw py::type_error(std::string(what) + " must be a sequence of 3-vectors"); }
            if (a.ndim() == 1 && a.shape(0) == 0) return std::make_pair(a, (size_t)0);
            if (a.ndim() != 2 || a.shape(1) != 3) throw py::type_error(std::string(what) + " must be a sequence of 3-vectors");
            return std::make_pair(a, (size_t)a.shape(0));
        };
        auto [xa, na] = to_xyz(coords_a, "coords_a");
        auto [xb, nb] = to_xyz(coords_b, "coords_b");
        if (na != nb)
            throw py::value_error("Expected matrices with the same length, got lengths " + std::to_string(na) + " and " + std::to_string(nb) + "!");
        a.wf = resolve_keys(keys, na);
        a.xa = xa; a.xb = xb; a.n = na;
        if (na == 0) return a;
        if (a.sa.size() < na || a.sb.size() < nb) throw py::value_error("The category sequences are shorter than the coordinate lists!");
        return a;
    }

    std::vector<double> from_coords(const py::object& seq_a, const py::object& seq_b, const py::object& coords_a,
                                    const py::object& coords_b, const std::optional<std::vector<std::string>>& keys) {
        const CoordsCall a = coords_call(seq_a, seq_b, coords_a, coords_b, keys);
        if (a.n == 0) return {};
        const auto d = ensure_ctx();
        const size_t n_pts = a.n;
        const double *pa = a.xa.data(), *pb = a.xb.data();
        return score_rows(d, n_pts, a.wf, [&](locohd_ctx* c, locohd_envset** ea, locohd_envset** eb) {
            int st = locohd_envset_from_coords(c, n_pts, pa, a.sa.data(), ea);
            if (!st) st = locohd_envset_from_coords(c, n_pts, pb, a.sb.data(), eb);
            return st;
        });
    }

    // from_coords with the coordinate gradients of the scores: (scores [n], grad_a [n, 3], grad_b [n, 3]),
    // grad = sum_r pair_weights[r] dS_r/dxyz (pair_weights None: all 1)
    py::tuple from_coords_grad(const py::object& seq_a, const py::object& seq_b, const py::object& coords_a,
                               const py::object& coords_b, const std::optional<std::vector<std::string>>& keys,
                               const py::object& pair_weights) {
        const CoordsCall a = coords_call(seq_a, seq_b, coords_a, coords_b, keys);
        const size_t n = a.n;
        F64Array pw;
        const double* w = weights_of(pair_weights, n, pw);
        py::array_t<double> out(n), ga({(py::ssize_t)n, (py::ssize_t)3}), gb({(py::ssize_t)n, (py::ssize_t)3});
        if (n) {
            const auto d = ensure_ctx();
            double *o = out.mutable_data(), *pga = ga.mutable_data(), *pgb = gb.mutable_data();
            device_call(d, [&](locohd_ctx* c) {
                return locohd_from_coords_grad(c, n, a.xa.data(), a.sa.data(), a.xb.data(), a.sb.data(),
                                               a.wf.empty() ? nullptr : a.wf.data(), w, o, pga, pgb);
            });
        }
        return py::make_tuple(out, ga, gb);
    }

    // ---- from_primitives (locohd.rs:479-567)
    struct Flat {
        std::vector<double> xyz;
        std::vector<uint16_t> cat;
        std::vector<uint32_t> tag;
    };
    static const PrimitiveAtom& as_atom(PyObject* item) {   // subclasses etc.; anything else is a TypeError, as with PyO3
        try {
            return py::handle(item).cast<const PrimitiveAtom&>();
        } catch (const py::cast_error&) {
            throw py::type_error("'" + std::string(Py_TYPE(item)->tp_name) + "' object cannot be converted to 'PrimitiveAtom'");
        }
    }
    Flat flatten(const py::handle& prims, const char* what) {
        if (py::isinstance<py::str>(prims)) throw py::type_error(std::string(what) + ": can't extract `str` to a list");
        Flat f;
        const py::ssize_t hint = py::len_hint(prims);
        if (hint > 0) { f.xyz.reserve(3 * hint); f.cat.reserve(hint); f.tag.reserve(hint); }
        // consecutive primitives usually share their tag (one tag per residue) and often their type: compare with
        // the previous strings before looking anything up.  For lists / tuples the previous item stays alive (the
        // container holds it), so the comparison goes through pointers; for other iterables the previous strings are
        // kept BY VALUE (a generator's previous item may already be gone when the next one arrives).
        const std::string *prev_tag = nullptr, *prev_type = nullptr;
        std::string last_tag, last_type;
        uint32_t last_tag_id = 0;
        uint16_t last_cat = 0;
        auto take = [&](const PrimitiveAtom& p, bool stays_alive) {
            f.xyz.push_back(p.coordinates[0]); f.xyz.push_back(p.coordinates[1]); f.xyz.push_back(p.coordinates[2]);
            if (!prev_type || *prev_type != p.primitive_type) {
                last_cat = cat_id(p.primitive_type);
                if (stays_alive) prev_type = &p.primitive_type; else { last_type = p.primitive_type; prev_type = &last_type; }
            }
            if (!prev_tag || *prev_tag != p.tag) {
                last_tag_id = intern_tag(p.tag);
                if (stays_alive) prev_tag = &p.tag; else { last_tag = p.tag; prev_tag = &last_tag; }
            }
            f.cat.push_back(last_cat);
            f.tag.push_back(last_tag_id);
        };
        // Fast path for what callers pass in practice - a list (or tuple) of exact PrimitiveAtom instances: no iterator
        // protocol, and the C++ object is taken from the instance directly instead of through the generic caster
        // (the reference clones every atom at this point, locohd.rs:480-481; here the cost is ~25 ns per atom).
        static PyTypeObject* const atom_type = reinterpret_cast<PyTypeObject*>(py::type::of<PrimitiveAtom>().ptr());
        auto fast = [&](PyObject* item, bool stays_alive) -> bool {
            if (Py_TYPE(item) != atom_type) return false;
            auto* inst = reinterpret_cast<py::detail::instance*>(item);
            const auto* p = static_cast<const PrimitiveAtom*>(inst->get_value_and_holder().value_ptr());
            if (!p) return false;
            take(*p, stays_alive);
            return true;
        };
        PyObject* seq = prims.ptr();
        if (PyList_CheckExact(seq) || PyTuple_CheckExact(seq)) {
            const Py_ssize_t n = PySequence_Fast_GET_SIZE(seq);
            for (Py_ssize_t k = 0; k < n; ++k) {
                PyObject* item = PySequence_Fast_GET_ITEM(seq, k);   // borrowed; the GIL is held and nothing below runs Python code
                if (!fast(item, true)) take(as_atom(item), true);
            }
            return f;
        }
        for (auto item : prims)
            if (!fast(item.ptr(), false)) take(as_atom(item.ptr()), false);
        return f;
    }

    std::vector<double> from_primitives(const py::object& prim_a, const py::object& prim_b, const py::object& anchor_pairs,
                                        double threshold) {
        // AnchorPairSpecifier (locohd.rs:34-40): a list of (i, j, key) triples is tried first, then (i, j) pairs;
        // an empty list therefore counts as "with keys".
        if (py::isinstance<py::str>(anchor_pairs)) throw py::type_error("anchor_pairs: can't extract `str` to a list");
        std::vector<uint32_t> anchors;
        std::vector<std::string> key_list;
        bool with_keys = true, first = true;
        size_t n_pairs = 0;
        for (auto item : anchor_pairs) {
            long long i, j;
            if (PyTuple_CheckExact(item.ptr()) && PyTuple_GET_SIZE(item.ptr()) == 2 && (first || !with_keys) &&
                PyLong_CheckExact(PyTuple_GET_ITEM(item.ptr(), 0)) && PyLong_CheckExact(PyTuple_GET_ITEM(item.ptr(), 1))) {
                // fast path: a plain (int, int) tuple
                if (first) { with_keys = false; first = false; }
                i = PyLong_AsLongLong(PyTuple_GET_ITEM(item.ptr(), 0));
                j = PyLong_AsLongLong(PyTuple_GET_ITEM(item.ptr(), 1));
                if ((i == -1 || j == -1) && PyErr_Occurred()) throw py::error_already_set();
                if (i < 0 || j < 0) throw py::value_error("anchor indices must be non-negative");
                if (i > 0xFFFFFFFELL || j > 0xFFFFFFFELL) throw py::value_error("anchor index out of range");
                anchors.push_back((uint32_t)i); anchors.push_back((uint32_t)j);
                ++n_pairs;
                continue;
            }
            py::sequence t = py::reinterpret_borrow<py::sequence>(item);
            if (!PySequence_Check(item.ptr()) || py::isinstance<py::str>(item)) throw py::type_error("anchor_pairs must contain (int, int) or (int, int, str) tuples");
            const size_t len = t.size();
            if (first) { with_keys = (len == 3); first = false; }
            if (len != (with_keys ? 3u : 2u)) throw py::type_error("anchor_pairs must contain (int, int) or (int, int, str) tuples");
            i = t[0].cast<long long>(); j = t[1].cast<long long>();
            if (i < 0 || j < 0) throw py::value_error("anchor indices must be non-negative");
            if (i > 0xFFFFFFFELL || j > 0xFFFFFFFELL) throw py::value_error("anchor index out of range");
            anchors.push_back((uint32_t)i); anchors.push_back((uint32_t)j);
            if (with_keys) key_list.push_back(t[2].cast<std::string>());
            ++n_pairs;
        }
        std::optional<std::vector<std::string>> keys;
        if (with_keys) keys = std::move(key_list);
        const auto wf = resolve_keys(keys, n_pairs);
        if (n_pairs == 0) return {};
        // (tag ids come from one table per instance; the rule's pairs are translated through the same table when the
        //  context is created, so the order of the two steps does not matter)
        const Flat a = flatten(prim_a, "prim_a"), b = flatten(prim_b, "prim_b");
        const auto d = ensure_ctx();
        for (size_t k = 0; k < n_pairs; ++k)  // prim_seq[anchor_idx] panics upstream (locohd.rs:521)
            if (anchors[2 * k] >= a.cat.size() || anchors[2 * k + 1] >= b.cat.size())
                throw py::value_error("Anchor index out of range: pair " + std::to_string(k) + " = (" + std::to_string(anchors[2 * k]) +
                                      ", " + std::to_string(anchors[2 * k + 1]) + ")");
        std::vector<double> out(n_pairs);
        device_call(d, [&](locohd_ctx* c) {
            return locohd_from_primitives(c, a.cat.size(), a.xyz.data(), a.cat.data(), a.tag.data(), b.cat.size(),
                                          b.xyz.data(), b.cat.data(), b.tag.data(), n_pairs, anchors.data(),
                                          wf.empty() ? nullptr : wf.data(), threshold, out.data());
        });
        return out;
    }

    // ---- array API (SURVEY.md §8(f) N1): integer category / tag ids and an [n, 3] coordinate array per structure.
    // Tag ids are opaque integers for a rule without a list; with a tag-pair list they must come from intern_tags(),
    // which maps strings to the ids the rule's pairs were interned with.
    std::vector<uint32_t> wf_indices(const py::object& wf_idx, size_t n) const {
        std::vector<uint32_t> wf;
        if (!wf_idx.is_none()) {
            wf = wf_idx.cast<std::vector<uint32_t>>();
            if (wf.size() != n) throw py::value_error("wf_idx must have one entry per anchor pair");
            for (uint32_t w : wf) if (w >= wfs.size()) throw py::value_error("wf_idx entry out of range");
        }
        return wf;
    }

    py::array_t<uint32_t> intern_tags(const py::object& tags) {
        const auto names = to_strings(tags, "tags");
        py::array_t<uint32_t> out(names.size());
        auto* o = out.mutable_data();
        for (size_t i = 0; i < names.size(); ++i) o[i] = intern_tag(names[i]);
        return out;
    }

    // list[PrimitiveAtom] -> (xyz [n, 3] float64, category ids uint16, tag ids uint32): the arrays from_arrays,
    // structures and Structures.update_xyz take; converts a structure once instead of on every call
    py::tuple to_arrays(const py::object& prims) {
        const Flat f = flatten(prims, "primitives");
        const size_t n = f.cat.size();
        py::array_t<double> xyz({(py::ssize_t)n, (py::ssize_t)3});
        std::copy(f.xyz.begin(), f.xyz.end(), xyz.mutable_data());
        py::array_t<uint16_t> cat(n);
        std::copy(f.cat.begin(), f.cat.end(), cat.mutable_data());
        py::array_t<uint32_t> tag(n);
        std::copy(f.tag.begin(), f.tag.end(), tag.mutable_data());
        return py::make_tuple(xyz, cat, tag);
    }

    py::array_t<uint16_t> category_ids(const py::object& types) const {
        const auto names = to_strings(types, "primitive types");
        py::array_t<uint16_t> out(names.size());
        auto* o = out.mutable_data();
        for (size_t i = 0; i < names.size(); ++i) o[i] = cat_id(names[i]);
        return out;
    }

    static size_t check_arrays(const F64Array& xyz_a, const U16Array& cat_a, const U32Array& tag_a, const F64Array& xyz_b,
                               const U16Array& cat_b, const U32Array& tag_b, const U32Array& anchors) {
        const size_t na = cat_a.size(), nb = cat_b.size();
        if ((size_t)xyz_a.size() != 3 * na || (size_t)tag_a.size() != na || (size_t)xyz_b.size() != 3 * nb || (size_t)tag_b.size() != nb)
            throw py::value_error("xyz must be [n, 3], category and tag [n]");
        if (anchors.size() % 2) throw py::value_error("anchors must be [n_pairs, 2]");
        return anchors.size() / 2;
    }

    py::array_t<double> from_arrays(F64Array xyz_a, U16Array cat_a, U32Array tag_a, F64Array xyz_b, U16Array cat_b,
                                    U32Array tag_b, U32Array anchors, double threshold, const py::object& wf_idx) {
        const size_t na = cat_a.size(), nb = cat_b.size();
        const size_t P = check_arrays(xyz_a, cat_a, tag_a, xyz_b, cat_b, tag_b, anchors);
        const auto wf = wf_indices(wf_idx, P);
        py::array_t<double> out(P);
        const auto d = ensure_ctx();
        double* o = out.mutable_data();
        device_call(d, [&](locohd_ctx* c) {
            return locohd_from_primitives(c, na, xyz_a.data(), cat_a.data(), tag_a.data(), nb, xyz_b.data(), cat_b.data(),
                                          tag_b.data(), P, anchors.data(), wf.empty() ? nullptr : wf.data(), threshold, o);
        });
        return out;
    }

    // from_arrays with the coordinate gradients of the scores: (scores [P], grad_a [n_a, 3], grad_b [n_b, 3]),
    // grad = sum_p pair_weights[p] dS_p/dxyz (pair_weights None: all 1)
    py::tuple from_arrays_grad(F64Array xyz_a, U16Array cat_a, U32Array tag_a, F64Array xyz_b, U16Array cat_b,
                               U32Array tag_b, U32Array anchors, double threshold, const py::object& wf_idx,
                               const py::object& pair_weights) {
        const size_t na = cat_a.size(), nb = cat_b.size();
        const size_t P = check_arrays(xyz_a, cat_a, tag_a, xyz_b, cat_b, tag_b, anchors);
        const auto wf = wf_indices(wf_idx, P);
        F64Array pw;
        if (!pair_weights.is_none()) {
            pw = pair_weights.cast<F64Array>();
            if ((size_t)pw.size() != P) throw py::value_error("pair_weights must have one entry per anchor pair");
        }
        py::array_t<double> out(P), ga({(py::ssize_t)na, (py::ssize_t)3}), gb({(py::ssize_t)nb, (py::ssize_t)3});
        const auto d = ensure_ctx();
        double *o = out.mutable_data(), *pga = ga.mutable_data(), *pgb = gb.mutable_data();
        device_call(d, [&](locohd_ctx* c) {
            return locohd_from_primitives_grad(c, na, xyz_a.data(), cat_a.data(), tag_a.data(), nb, xyz_b.data(),
                                               cat_b.data(), tag_b.data(), P, anchors.data(), wf.empty() ? nullptr : wf.data(),
                                               threshold, pair_weights.is_none() ? nullptr : pw.data(), o, pga, pgb);
        });
        return py::make_tuple(out, ga, gb);
    }

    // ---- resident batches (SURVEY.md §8(f) N1 / N4): what the callers loop over upstream - one reference against
    // many models (casp14_extend_with_locohd.py:58-79), frame 0 against every frame (trajectory_analyzer.py:112-120),
    // all pairs of an ensemble (compare_ensembles.py:273-296) - with the structures uploaded once.
    std::shared_ptr<Structures> structures(const U64Array& offsets, const py::array& xyz, const U16Array& cat,
                                           const U32Array& tag) {
        if (offsets.size() < 2) throw py::value_error("prim_offsets must hold n_structures + 1 entries");
        const uint64_t n_structs = (uint64_t)offsets.size() - 1;
        const uint64_t n = offsets.data()[n_structs];
        if ((uint64_t)xyz.size() != 3 * n || (uint64_t)cat.size() != n || (uint64_t)tag.size() != n)
            throw py::value_error("xyz must be [n, 3], category and tag [n] with n = prim_offsets[-1]");
        auto s = std::make_shared<Structures>();
        s->dev = ensure_ctx();
        s->n_structs = n_structs; s->n_prims = n;
        s->offsets.assign(offsets.data(), offsets.data() + offsets.size());
        if (py::isinstance<py::array_t<float>>(xyz)) {
            auto a = py::array_t<float, py::array::c_style | py::array::forcecast>::ensure(xyz);
            device_call(s->dev, [&](locohd_ctx* c) {
                return locohd_structs_create_f32(c, n_structs, offsets.data(), a.data(), cat.data(), tag.data(), &s->h);
            });
        } else {
            auto a = F64Array::ensure(xyz);
            if (!a) throw py::type_error("xyz must be a float array");
            device_call(s->dev, [&](locohd_ctx* c) {
                return locohd_structs_create(c, n_structs, offsets.data(), a.data(), cat.data(), tag.data(), &s->h);
            });
        }
        return s;
    }

    std::shared_ptr<Environments> environments(const std::shared_ptr<Structures>& st, const U32Array& anchor_prim,
                                               double threshold, const py::object& anchor_struct) {
        if (!st) throw py::value_error("structures is None");
        st->need();
        const auto d = ensure_ctx();
        if (d != st->dev) throw py::value_error("the structures were uploaded for another device / context");
        const uint64_t n = (uint64_t)anchor_prim.size();
        U32Array as;
        const uint32_t* as_ptr = nullptr;
        if (!anchor_struct.is_none()) {
            as = U32Array::ensure(anchor_struct);
            if (!as || (uint64_t)as.size() != n) throw py::value_error("anchor_struct must have one entry per anchor");
            as_ptr = as.data();
        }
        auto e = std::make_shared<Environments>();
        e->dev = d;
        e->n_env = n;
        device_call(d, [&](locohd_ctx* c) {
            return locohd_envset_build(c, st->h, n, as_ptr, anchor_prim.data(), threshold, 0, &e->h);
        });
        return e;
    }

    // jobs: [n_jobs, 3] (first environment in env_a, first environment in env_b, number of anchor pairs).
    // reduce: None -> per-anchor scores of all jobs, concatenated; or any of "job_mean", "anchor_mean", "anchor_std"
    // (a string or a sequence of them; "scores" may be listed too) -> dict of arrays, reduced on the device.
    py::object score_batch(const std::shared_ptr<Environments>& ea, const std::shared_ptr<Environments>& eb,
                           const U64Array& jobs, const py::object& reduce, const py::object& wf_idx) {
        if (!ea || !eb || !ea->h || !eb->h) throw py::value_error("environments are None or closed");
        if (ea->dev != eb->dev) throw py::value_error("the two environment sets live in different contexts");
        if (jobs.ndim() != 2 || jobs.shape(1) != 3) throw py::value_error("jobs must be [n_jobs, 3]: (a_first, b_first, n)");
        const uint64_t n_jobs = (uint64_t)jobs.shape(0);
        std::vector<locohd_job> hj(n_jobs);
        uint64_t total = 0;
        for (uint64_t j = 0; j < n_jobs; ++j) {
            hj[j] = locohd_job{jobs.data()[3 * j], jobs.data()[3 * j + 1], jobs.data()[3 * j + 2]};
            total += hj[j].n;
        }
        const auto wf = wf_indices(wf_idx, total);
        bool want_scores = reduce.is_none(), want_jm = false, want_am = false, want_as = false;
        if (!reduce.is_none()) {
            std::vector<std::string> names;
            if (py::isinstance<py::str>(reduce)) names.push_back(reduce.cast<std::string>());
            else names = to_strings(reduce, "reduce");
            for (const auto& nme : names) {
                if (nme == "scores") want_scores = true;
                else if (nme == "job_mean") want_jm = true;
                else if (nme == "anchor_mean") want_am = true;
                else if (nme == "anchor_std") want_as = true;
                else throw py::value_error("reduce: unknown name \"" + nme + "\" (scores, job_mean, anchor_mean, anchor_std)");
            }
        }
        const uint64_t n_anchor = n_jobs ? hj[0].n : 0;
        py::array_t<double> scores(want_scores ? total : 0), jm(want_jm ? n_jobs : 0), am(want_am ? n_anchor : 0),
            as(want_as ? n_anchor : 0);
        double *ps = want_scores ? scores.mutable_data() : nullptr, *pj = want_jm ? jm.mutable_data() : nullptr,
               *pm = want_am ? am.mutable_data() : nullptr, *pd = want_as ? as.mutable_data() : nullptr;
        if (total)
            device_call(ea->dev, [&](locohd_ctx* c) {
                return locohd_score_jobs_stats(c, ea->h, eb->h, n_jobs, hj.data(), wf.empty() ? nullptr : wf.data(), ps, pj, pm, pd);
            });
        if (reduce.is_none()) return scores;
        py::dict out;
        if (want_scores) out["scores"] = scores;
        if (want_jm) out["job_mean"] = jm;
        if (want_am) out["anchor_mean"] = am;
        if (want_as) out["anchor_std"] = as;
        return out;
    }
};

}  // namespace

PYBIND11_MODULE(loco_hd, m) {
    m.doc() = "B200-native LoCoHD host module: the reference's PyO3 classes over the CUDA C ABI (no CPU scoring path)";
    m.attr("ABI_VERSION") = locohd_abi_version();
    m.def("device_count", &locohd_device_count, "Number of visible CUDA devices");
    m.def("set_device", [](int d) { g_device = d; }, py::arg("device"),
          "GPU used by LoCoHD instances for their next scoring call (default: $LOCOHD_DEVICE or 0)");
    m.def("get_device", &default_device);

    py::class_<WeightFunction>(m, "WeightFunction")
        .def(py::init<std::string, std::vector<double>>(), py::arg("function_name"), py::arg("parameters"))
        .def_readonly("parameters", &WeightFunction::parameters)
        .def_readonly("function_name", &WeightFunction::function_name)
        .def("integral_point", &WeightFunction::integral_point, py::arg("point"))
        .def("integral_vec", &WeightFunction::integral_vec, py::arg("points"))
        .def("integral_range", &WeightFunction::integral_range, py::arg("point_from"), py::arg("point_to"));

    py::class_<PrimitiveAtom>(m, "PrimitiveAtom")
        .def(py::init([](std::string t, std::string tag, std::array<double, 3> c) {
                 return PrimitiveAtom{std::move(t), std::move(tag), c};
             }),
             py::arg("primitive_type"), py::arg("tag"), py::arg("coordinates"))
        .def_readwrite("primitive_type", &PrimitiveAtom::primitive_type)
        .def_readwrite("tag", &PrimitiveAtom::tag)
        .def_property(
            "coordinates", [](const PrimitiveAtom& p) { return std::vector<double>(p.coordinates.begin(), p.coordinates.end()); },
            [](PrimitiveAtom& p, std::array<double, 3> c) { p.coordinates = c; });

    py::class_<TagPairingRule>(m, "TagPairingRule")
        .def(py::init<const py::dict&>(), py::arg("variant"))
        .def("pair_accepted", &TagPairingRule::pair_accepted, py::arg("pair"))
        .def("get_dbg_str", &TagPairingRule::dbg);

    py::class_<StatisticalDistance>(m, "StatisticalDistance")
        .def(py::init<std::string, std::vector<double>>(), py::arg("distance_name"), py::arg("parameters"))
        .def("run", &StatisticalDistance::run, py::arg("p1"), py::arg("p2"));

    py::class_<LoCoHD>(m, "LoCoHD")
        .def(py::init<const py::object&, const py::object&, const py::object&, const py::object&, const py::object&,
                      const py::object&>(),
             py::arg("categories"), py::arg("w_func") = py::none(), py::arg("tag_pairing_rule") = py::none(),
             py::arg("n_of_threads") = py::none(), py::arg("category_weights") = py::none(),
             py::arg("statistical_distance") = py::none())
        .def_property_readonly("categories", &LoCoHD::categories_dict)
        .def_property_readonly("category_weights", [](const LoCoHD& l) { return l.category_weights; })
        .def_property_readonly("w_func", &LoCoHD::w_func_object)
        .def_property_readonly("tag_pairing_rule", [](const LoCoHD& l) { return l.rule; })
        .def("from_anchors", &LoCoHD::from_anchors, py::arg("seq_a"), py::arg("seq_b"), py::arg("dists_a"),
             py::arg("dists_b"), py::arg("w_func_key") = py::none())
        .def("from_dmxs", &LoCoHD::from_dmxs, py::arg("seq_a"), py::arg("seq_b"), py::arg("dmx_a"), py::arg("dmx_b"),
             py::arg("w_func_keys") = py::none())
        .def("from_coords", &LoCoHD::from_coords, py::arg("seq_a"), py::arg("seq_b"), py::arg("coords_a"),
             py::arg("coords_b"), py::arg("w_func_keys") = py::none())
        .def("from_dmxs_grad", &LoCoHD::from_dmxs_grad, py::arg("seq_a"), py::arg("seq_b"), py::arg("dmx_a"),
             py::arg("dmx_b"), py::arg("w_func_keys") = py::none(), py::arg("pair_weights") = py::none(),
             "from_dmxs with the gradients of the scores with respect to every matrix entry (an extension)")
        .def("from_coords_grad", &LoCoHD::from_coords_grad, py::arg("seq_a"), py::arg("seq_b"), py::arg("coords_a"),
             py::arg("coords_b"), py::arg("w_func_keys") = py::none(), py::arg("pair_weights") = py::none(),
             "from_coords with the coordinate gradients of the scores (an extension)")
        .def("from_primitives", &LoCoHD::from_primitives, py::arg("prim_a"), py::arg("prim_b"), py::arg("anchor_pairs"),
             py::arg("threshold_distance"))
        .def("from_arrays", &LoCoHD::from_arrays, py::arg("xyz_a"), py::arg("cat_a"), py::arg("tag_a"), py::arg("xyz_b"),
             py::arg("cat_b"), py::arg("tag_b"), py::arg("anchors"), py::arg("threshold_distance"),
             py::arg("wf_idx") = py::none(),
             "Array form of from_primitives: integer category ids (index into `categories`, 0xFFFF = unknown; see "
             "category_ids), integer tag ids (opaque for a rule without a tag list, from intern_tags otherwise), "
             "[n, 3] float64 coordinates, [n_pairs, 2] anchor indices.  Returns a float64 array.")
        .def("from_arrays_grad", &LoCoHD::from_arrays_grad, py::arg("xyz_a"), py::arg("cat_a"), py::arg("tag_a"),
             py::arg("xyz_b"), py::arg("cat_b"), py::arg("tag_b"), py::arg("anchors"), py::arg("threshold_distance"),
             py::arg("wf_idx") = py::none(), py::arg("pair_weights") = py::none(),
             "from_arrays with the coordinate gradients of the scores (an extension): returns (scores [n_pairs], "
             "grad_a [n_a, 3], grad_b [n_b, 3]) with grad = sum_p pair_weights[p] dS_p/dxyz (None: all 1).  At tied "
             "distances the gradient is one-sided; threshold crossings are not differentiated.")
        .def("intern_tags", &LoCoHD::intern_tags, py::arg("tags"),
             "Tag strings -> the uint32 ids this instance uses for them (the ids of a WithList rule's tag pairs included).")
        .def("to_arrays", &LoCoHD::to_arrays, py::arg("primitives"),
             "list[PrimitiveAtom] -> (xyz [n, 3] float64, category ids uint16, tag ids uint32) for from_arrays / structures.")
        .def("category_ids", &LoCoHD::category_ids, py::arg("primitive_types"),
             "Primitive type names -> uint16 category ids (0xFFFF for a name that is not in `categories`).")
        .def("structures", &LoCoHD::structures, py::arg("prim_offsets"), py::arg("xyz"), py::arg("categories"), py::arg("tags"),
             "Upload a set of structures once: structure s owns primitives [prim_offsets[s], prim_offsets[s + 1]) of the "
             "concatenated arrays (float32 coordinates travel as float32 and are widened on the device).")
        .def("environments", &LoCoHD::environments, py::arg("structures"), py::arg("anchor_prim"), py::arg("threshold_distance"),
             py::arg("anchor_struct") = py::none(),
             "Sorted environments of a list of anchors (structure anchor_struct[e], default 0; primitive anchor_prim[e]).")
        .def("score_batch", &LoCoHD::score_batch, py::arg("env_a"), py::arg("env_b"), py::arg("jobs"),
             py::arg("reduce") = py::none(), py::arg("wf_idx") = py::none(),
             "Score runs of identity-paired environments: jobs is [n_jobs, 3] (a_first, b_first, n).  reduce=None returns "
             "the per-anchor scores; \"job_mean\", \"anchor_mean\", \"anchor_std\" (or a list of them, optionally with "
             "\"scores\") are reduced on the device and returned in a dict.");

    py::class_<Structures, std::shared_ptr<Structures>>(m, "Structures")
        .def_readonly("n_structures", &Structures::n_structs)
        .def_readonly("n_primitives", &Structures::n_prims)
        .def_property_readonly("prim_offsets", [](const Structures& s) { return s.offsets; })
        .def("update_xyz", &Structures::update_xyz, py::arg("xyz"), "Replace all coordinates (same topology: trajectory frames).")
        .def("update_from_atoms", &Structures::update_from_atoms, py::arg("atom_xyz"), py::arg("segment_start"),
             py::arg("atom_index"), py::arg("first_structure") = 0,
             "Frames of one compiled topology: float32 atom coordinates [n_frames, n_atoms, 3] -> primitive centroids of "
             "structures first_structure ... on the device (PrimitiveAssigner.compile_topology gives the index arrays).")
        .def("close", &Structures::close);

    py::class_<Environments, std::shared_ptr<Environments>>(m, "Environments")
        .def("__len__", [](const Environments& e) { return e.n_env; })
        .def("close", &Environments::close);
}
