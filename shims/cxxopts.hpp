// shims/cxxopts.hpp -- minimal from-scratch stand-in for the subset of the cxxopts 3.x API that the
// reference's simple_trainer.cpp:26-62 uses (Options, add_options()(...) chains, value<T>()->default_value,
// parse, count, operator[]().as<T>(), help).  cxxopts itself is a FetchContent dependency of the
// reference (CMakeLists.txt) that is not available offline; this shim exists ONLY so that the unchanged
// simple_trainer.cpp can be compiled against the gsplat_b200 operator layer (oracle/build_simple_trainer.py).
#pragma once
#include <map>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

namespace cxxopts {

class Value {
public:
    std::shared_ptr<Value> default_value(const std::string &v) {
        def_ = v;
        has_def_ = true;
        return self_.lock();
    }
    bool has_default() const { return has_def_; }
    const std::string &get_default() const { return def_; }
    std::weak_ptr<Value> self_;

private:
    std::string def_;
    bool has_def_ = false;
};

template <typename T>
std::shared_ptr<Value> value() {
    auto v = std::make_shared<Value>();
    v->self_ = v;
    return v;
}

class OptionValue {
public:
    OptionValue() = default;
    explicit OptionValue(std::string s) : text_(std::move(s)) {}
    template <typename T>
    T as() const {
        std::istringstream is(text_);
        T out{};
        if constexpr (std::is_same<T, std::string>::value) {
            return text_;
        } else {
            is >> out;
            if (is.fail()) throw std::runtime_error("cannot parse option value '" + text_ + "'");
            return out;
        }
    }

private:
    std::string text_;
};

class ParseResult {
public:
    size_t count(const std::string &name) const {
        auto it = counts_.find(name);
        return it == counts_.end() ? 0 : it->second;
    }
    OptionValue operator[](const std::string &name) const {
        auto it = values_.find(name);
        if (it == values_.end()) throw std::runtime_error("option '" + name + "' has no value");
        return OptionValue(it->second);
    }
    std::map<std::string, size_t> counts_;
    std::map<std::string, std::string> values_;
};

class Options;

class OptionAdder {
public:
    explicit OptionAdder(Options &o) : opts_(o) {}
    OptionAdder &operator()(const std::string &names, const std::string &desc,
                            std::shared_ptr<Value> val = nullptr);

private:
    Options &opts_;
};

class Options {
public:
    Options(std::string program, std::string help) : program_(std::move(program)), help_(std::move(help)) {}
    OptionAdder add_options() { return OptionAdder(*this); }

    ParseResult parse(int argc, char **argv) {
        ParseResult r;
        for (auto &o : opts_)
            if (o.val && o.val->has_default()) r.values_[o.long_name] = o.val->get_default();
        for (int i = 1; i < argc; ++i) {
            std::string a = argv[i], name, val;
            bool has_val = false;
            if (a.rfind("--", 0) == 0) {
                name = a.substr(2);
                auto eq = name.find('=');
                if (eq != std::string::npos) {
                    val = name.substr(eq + 1);
                    name = name.substr(0, eq);
                    has_val = true;
                }
            } else if (a.size() == 2 && a[0] == '-') {
                name = resolve_short(a[1]);
            } else {
                throw std::runtime_error("unexpected argument '" + a + "'");
            }
            const Opt *o = find(name);
            if (!o) throw std::runtime_error("unknown option '" + a + "'");
            if (o->val) {
                if (!has_val) {
                    if (i + 1 >= argc) throw std::runtime_error("option '" + a + "' needs a value");
                    val = argv[++i];
                }
                r.values_[o->long_name] = val;
            }
            r.counts_[o->long_name] += 1;
        }
        return r;
    }

    std::string help() const {
        std::ostringstream os;
        os << help_ << "\nUsage:\n  " << program_ << " [OPTION...]\n\n";
        for (auto &o : opts_) {
            os << "  ";
            if (o.short_name) os << "-" << o.short_name << ", ";
            os << "--" << o.long_name;
            if (o.val) os << " arg";
            os << "  " << o.desc;
            if (o.val && o.val->has_default()) os << " (default: " << o.val->get_default() << ")";
            os << "\n";
        }
        return os.str();
    }

    void add(const std::string &names, const std::string &desc, std::shared_ptr<Value> val) {
        Opt o;
        auto comma = names.find(',');
        if (comma != std::string::npos) {
            o.short_name = names[0];
            o.long_name = names.substr(comma + 1);
        } else {
            o.long_name = names;
        }
        o.desc = desc;
        o.val = std::move(val);
        opts_.push_back(o);
    }

private:
    struct Opt {
        char short_name = 0;
        std::string long_name, desc;
        std::shared_ptr<Value> val;
    };
    const Opt *find(const std::string &n) const {
        for (auto &o : opts_)
            if (o.long_name == n) return &o;
        return nullptr;
    }
    std::string resolve_short(char c) const {
        for (auto &o : opts_)
            if (o.short_name == c) return o.long_name;
        return std::string(1, c);
    }
    std::string program_, help_;
    std::vector<Opt> opts_;
};

inline OptionAdder &OptionAdder::operator()(const std::string &names, const std::string &desc,
                                            std::shared_ptr<Value> val) {
    opts_.add(names, desc, std::move(val));
    return *this;
}

}  // namespace cxxopts
