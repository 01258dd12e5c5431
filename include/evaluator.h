/* Drop-in for the reference's Source/evaluator.h (class Evaluator, evaluator.h:24-86) on top of the C ABI (mcb.h).
 *
 * Same class name, same public signatures, same error convention (bool returns; only Evaluator(std::string) throws),
 * so main.cpp:11-20 and drawer.cpp:828-831,925-936 compile against it unchanged.  What differs is where the work
 * happens: the equation is tokenised and lowered on the host once per set_equation(), and every evaluation runs on
 * the GPU through mcb_eval_points (there is no host evaluator behind this class).
 *
 * Observable behaviour kept from the reference:
 *   - Evaluator() holds "x+y" (evaluator.cpp:6-8); Evaluator(s) throws std::exception when s does not parse (:10-13);
 *   - set_equation(s) returns false on a parse error and the previous equation stays in force (evaluator.h:59 and
 *     SURVEY.md D6: the reference re-tokenises the stored good string on the next evaluate);
 *   - the grammar and the non-standard evaluation order are those of evaluator.cpp:22-237 (see csrc/mcb_lower.h).
 * Deliberate difference: equations the reference tokenizer accepts but then evaluates by reading outside its
 * operand stack ("x+", "-": undefined behaviour) are rejected.
 * The Win32 file dialogs of evaluator.cpp:240-332 are replaced by plain files: "equation.txt" in the working
 * directory (the dialogs' default name) or the path in $MCB_EQUATION_FILE.
 */
#pragma once

#include <cstdio>
#include <cstdlib>
#include <exception>
#include <iostream>
#include <string>

#include "mcb.h"

class Evaluator {
public:
    Evaluator() : ctx_(nullptr), equation_("x+y") {}
    explicit Evaluator(std::string s) : ctx_(nullptr), equation_("x+y") {
        if (!set_equation(s)) throw std::exception();
    }
    Evaluator(const Evaluator& o) : ctx_(nullptr), equation_(o.equation_), function_grammar_(o.function_grammar_) {}
    Evaluator& operator=(const Evaluator& o) {
        if (this != &o) {
            equation_ = o.equation_;
            function_grammar_ = o.function_grammar_;
            if (ctx_) { mcb_set_grammar(ctx_, grammar()); mcb_set_equation(ctx_, 0, equation_.c_str()); }
        }
        return *this;
    }
    ~Evaluator() { if (ctx_) mcb_destroy(ctx_); }

    bool set_equation(std::string s) {
        if (mcb_grammar_text(s.c_str(), grammar(), -1, nullptr, 0) != MCB_OK) return false; /* mcb_parse by default */
        std::string cleaned;
        for (char c : s) if (c != ' ') cleaned.push_back(c);
        equation_ = cleaned;
        if (ctx_ && mcb_set_equation(ctx_, 0, equation_.c_str()) != MCB_OK) return false;
        return true;
    }

    /* One point, on the GPU.  Field evaluation over a grid goes through Marching; this entry point exists because
     * the reference exposes it (Marching and tests call it), not because it is fast. */
    float evaluate(float x, float y, float z) {
        if (!ctx_) {
            if (mcb_create(device_from_env(), &ctx_) != MCB_OK) throw std::exception(); /* no CPU fallback */
            mcb_set_grammar(ctx_, grammar());
            if (mcb_set_equation(ctx_, 0, equation_.c_str()) != MCB_OK) throw std::exception();
        }
        const float p[3] = {x, y, z};
        float out = 0.f;
        if (mcb_eval_points(ctx_, 0, p, &out, 1, 0) != MCB_OK) throw std::exception();
        return out;
    }

    bool get_equation_from_file(std::string& str) {
        str = equation_;
        FILE* fp = std::fopen(file_name(), "r");
        if (!fp) return false;
        char buf[256];
        bool got = std::fgets(buf, sizeof buf, fp) != nullptr;
        std::fclose(fp);
        if (!got) return false;
        std::string line(buf);
        while (!line.empty() && (line.back() == '\n' || line.back() == '\r')) line.pop_back();
        if (!set_equation(line)) return false;
        str = line;
        return true;
    }
    bool save_equation_to_file() {
        if (equation_.empty()) return false;
        FILE* fp = std::fopen(file_name(), "w");
        if (!fp) return false;
        int ret = std::fprintf(fp, "%s", equation_.c_str());
        std::fclose(fp);
        return ret >= 0;
    }

    /* the reference's tokenizer self-test (evaluator.h:67-77) */
    void test() {
        check_parse("-(x+ -(y)* -.021)", 1); check_parse("(x(y)", 0); check_parse("(x)", 1); check_parse("(x-)", 0);
        check_parse("(-x)", 1); check_parse("-(-x)", 1); check_parse("", 0); check_parse("xyz", 1); check_parse("xy/z^-.22", 1);
    }
    void check_parse(std::string str, bool expect_success) {
        bool ok = mcb_parse(str.c_str()) == MCB_OK;
        if (ok == expect_success) std::cout << "PASS eq:" << str << std::endl;
        else std::cout << "FAIL eq:" << str << "\t expect " << expect_success << ", got " << ok << std::endl;
    }

    /* extension used by Marching: the current (cleaned) equation text */
    const std::string& equation() const { return equation_; }

    /* Extension: on = later set_equation calls accept sin( cos( sqrt( abs( and min(a,b) max(a,b) (MCB_GRAMMAR_FUNCTIONS, mcb.h); off (the
     * default) = exactly the reference's language.  The current equation is kept either way.  test() always checks the
     * reference grammar. */
    void set_function_grammar(bool on) {
        function_grammar_ = on;
        if (ctx_) mcb_set_grammar(ctx_, grammar());
    }
    int grammar() const { return function_grammar_ ? MCB_GRAMMAR_FUNCTIONS : MCB_GRAMMAR_REFERENCE; }

private:
    static int device_from_env() { const char* d = std::getenv("MCB_DEVICE"); return d ? std::atoi(d) : 0; }
    static const char* file_name() { const char* f = std::getenv("MCB_EQUATION_FILE"); return f ? f : "equation.txt"; }
    mcb_ctx* ctx_;
    std::string equation_;
    bool function_grammar_ = false;
};
