/* Host front end: tokenizer + symbolic two-stack execution + bytecode lowering.  See mcb_lower.h. */
#include "mcb_lower.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>

#include "../../include/mcb.h"

namespace mcb {

static inline bool is_operator(char c) { return c == '+' || c == '-' || c == '*' || c == '/' || c == '^'; }
static inline bool is_number(char c) { return (c >= '0' && c <= '9') || c == '.'; }
static inline bool is_variable(char c) { return (c >= 'x' && c <= 'z') || (c >= 'X' && c <= 'Z'); }

/* The function grammar's names, each spelt with its '(': the unary ones, then the two-argument min( and max(.  A name
 * is matched at a lowercase letter that is not a variable, so the x of max( is part of the name. */
static const int kNumFuncs = 6;
static const char* const kFuncNames[kNumFuncs] = {"sin(", "cos(", "sqrt(", "abs(", "min(", "max("};
static const char kFuncKinds[kNumFuncs] = {'S', 'C', 'Q', 'A', 'm', 'M'};
static inline bool two_args(int f) { return f >= 4; }

/* Accept/reject behaviour of evaluator.cpp:139-237, token for token; under GRAMMAR_FUNCTIONS a function name with its
 * '(' is one more kind of opening bracket, and a ',' separates the two arguments of min( / max(. */
bool tokenize(const std::string& eq_in, std::vector<Token>& out, std::string* cleaned, int grammar) {
    out.clear();
    if (eq_in.empty()) return false; /* evaluator.cpp:141 */
    std::string eq;
    for (char c : eq_in)
        if (c != ' ') eq.push_back(c); /* :147 — only blanks are stripped */

    enum { L_OP, L_NUM, L_VAR, L_BO, L_BC, L_NONE } last = L_NONE;
    bool neg = false;
    /* per open bracket: 0 plain or one argument, 1 two arguments before the ',', 2 two arguments after it */
    std::vector<char> open;
    for (size_t i = 0; i < eq.size(); i++) {
        char ch = eq[i];
        /* :162 unary minus; a ',' can only have been accepted under GRAMMAR_FUNCTIONS, where it acts as '(' does */
        if (ch == '-' && (i == 0 || eq[i - 1] == '(' || eq[i - 1] == ',' || is_operator(eq[i - 1]))) {
            if (neg) return false;
            neg = true;
            out.push_back({TOK_NEG, "NEG"});
            continue;
        }
        if (ch == '(') {
            if (last == L_VAR || last == L_NUM || last == L_BC) out.push_back({TOK_OP, "*"}); /* :172 implicit * */
            out.push_back({TOK_BRAC_O, "("});
            open.push_back(0);
            last = L_BO;
        } else if (ch == ')') {
            if (neg || last == L_BO || last == L_OP) return false; /* "-)", "()", "+)" */
            if (open.empty() || open.back() == 1) return false;   /* unbalanced, or min( / max( with one argument */
            out.push_back({TOK_BRAC_C, ")"});
            open.pop_back();
            last = L_BC;
        } else if (ch == ',' && grammar == GRAMMAR_FUNCTIONS) {
            if (neg || last == L_BO || last == L_OP) return false; /* the rules before ')': "min(,x)", "min(x+,y)" */
            if (open.empty() || open.back() != 1) return false;   /* only directly inside min( / max(, and only once */
            out.push_back({TOK_COMMA, ","});
            open.back() = 2;
            last = L_BO; /* the rules after '(' */
        } else if (is_operator(ch)) {
            if (neg || last == L_BO || last == L_OP || last == L_NONE) return false;
            out.push_back({TOK_OP, std::string(1, ch)});
            last = L_OP;
        } else if (is_number(ch)) {
            if (last == L_VAR || last == L_BC) out.push_back({TOK_OP, "*"}); /* :194 */
            std::string s(1, ch);
            bool dot = (ch == '.');
            while (i + 1 < eq.size() && is_number(eq[i + 1])) {
                if (eq[i + 1] == '.') {
                    if (dot) return false;
                    dot = true;
                }
                s.push_back(eq[++i]);
            }
            if (s == ".") return false;
            out.push_back({TOK_NUM, s});
            last = L_NUM;
        } else if (is_variable(ch)) {
            if (last == L_VAR || last == L_NUM || last == L_BC) out.push_back({TOK_OP, "*"}); /* :217 */
            out.push_back({TOK_VAR, std::string(1, ch)});
            last = L_VAR;
        } else if (grammar == GRAMMAR_FUNCTIONS && ch >= 'a' && ch <= 'z') {
            int f = 0;
            while (f < kNumFuncs && eq.compare(i, std::strlen(kFuncNames[f]), kFuncNames[f]) != 0) f++;
            if (f == kNumFuncs) return false; /* not a function name, or a name without its '(' */
            if (last == L_VAR || last == L_NUM || last == L_BC) out.push_back({TOK_OP, "*"}); /* as before '(' */
            out.push_back({TOK_FUNC, kFuncNames[f]});
            i += std::strlen(kFuncNames[f]) - 1; /* eq[i] is now the '(': the unary-minus rule sees it */
            open.push_back(two_args(f) ? 1 : 0);
            last = L_BO;
        } else {
            return false; /* :224 unknown character */
        }
        neg = false;
    }
    if (!open.empty()) return false;
    if (cleaned) *cleaned = eq;
    return true;
}

/* ------------------------------------------------------------------------------------------------------------ */

namespace {

struct Builder {
    Expr& e;
    std::map<std::tuple<char, int, int, uint32_t>, int> memo; /* hash-consing: equal subtrees share a node */
    explicit Builder(Expr& ex) : e(ex) {}
    int make(char kind, int a, int b, float v) {
        uint32_t bits;
        std::memcpy(&bits, &v, 4);
        auto key = std::make_tuple(kind, a, b, bits);
        auto it = memo.find(key);
        if (it != memo.end()) return it->second;
        Node n;
        n.kind = kind; n.a = a; n.b = b; n.value = v;
        if (kind == 'x') n.mask = 1;
        else if (kind == 'y') n.mask = 2;
        else if (kind == 'z') n.mask = 4;
        else if (kind == 'c') n.mask = 0;
        else if (b < 0) n.mask = e.nodes[a].mask; /* 'N' and the functions */
        else n.mask = e.nodes[a].mask | e.nodes[b].mask;
        e.nodes.push_back(n);
        memo[key] = (int)e.nodes.size() - 1;
        return (int)e.nodes.size() - 1;
    }
};

int precedence(char c) { /* evaluator.cpp:111-124 */
    switch (c) {
        case 'N': return 4;
        case '^': return 3;
        case '/': case '*': return 2;
        case '+': case '-': return 1;
        default: return 0; /* ( ) and the function markers: the look-back never crosses them */
    }
}
bool is_func(char c) { return c == 'S' || c == 'C' || c == 'Q' || c == 'A' || c == 'm' || c == 'M'; }
bool is_func2(char c) { return c == 'm' || c == 'M'; } /* min, max: two operands */

struct Machine {
    Builder& b;
    std::vector<char> ops;
    std::vector<int> vals;
    bool ok = true;
    explicit Machine(Builder& bb) : b(bb) {}
    int pop_val() {
        if (vals.empty()) { ok = false; return 0; }
        int v = vals.back(); vals.pop_back(); return v;
    }
    /* Evaluator::evaluate_op, evaluator.cpp:22-48 */
    void reduce() {
        if (!ok) return;
        if (ops.empty()) { ok = false; return; }
        char op = ops.back(); ops.pop_back();
        if (is_operator(op)) {
            int val1 = pop_val();
            if (!ops.empty() && precedence(ops.back()) > precedence(op)) reduce(); /* one-level look-back */
            int val2 = pop_val();
            if (!ok) return;
            vals.push_back(b.make(op, val2, val1, 0.f));
        } else if (op == 'N') {
            int v = pop_val();
            if (!ok) return;
            vals.push_back(b.make('N', v, -1, 0.f));
        } else {
            ok = false; /* a stray '(' or function marker — the reference throws (evaluator.cpp:47) */
        }
    }
};

} /* namespace */

bool build_expr(const std::vector<Token>& toks, Expr& e) { /* f(E) is (E) with f applied at the ')'; min(A,B) closes A at
                                                                the ',' as (A) and B at the ')' as (B) */
    e.nodes.clear();
    e.root = -1;
    Builder b(e);
    Machine m(b);
    for (const Token& t : toks) {
        switch (t.type) {
            case TOK_NEG: m.ops.push_back('N'); break;
            case TOK_VAR: {
                char c = t.text[0];
                char v = (c == 'x' || c == 'X') ? 'x' : (c == 'y' || c == 'Y') ? 'y' : 'z';
                m.vals.push_back(b.make(v, -1, -1, 0.f));
                break;
            }
            case TOK_NUM: {
                float v = std::strtof(t.text.c_str(), nullptr); /* stof, evaluator.cpp:82 */
                m.vals.push_back(b.make('c', -1, -1, v));
                break;
            }
            case TOK_BRAC_O: m.ops.push_back('('); break;
            case TOK_FUNC:
                for (int f = 0; f < kNumFuncs; f++)
                    if (t.text == kFuncNames[f]) m.ops.push_back(kFuncKinds[f]);
                break;
            case TOK_COMMA: /* the first argument is complete: reduce down to the marker, which stays */
                while (m.ok && !m.ops.empty() && m.ops.back() != '(' && !is_func(m.ops.back())) m.reduce();
                if (m.ops.empty() || !is_func2(m.ops.back())) m.ok = false;
                break;
            case TOK_BRAC_C:
                while (m.ok && !m.ops.empty() && m.ops.back() != '(' && !is_func(m.ops.back())) m.reduce();
                if (m.ops.empty()) m.ok = false;
                else {
                    const char f = m.ops.back();
                    m.ops.pop_back();
                    if (is_func2(f) && m.ok) {
                        const int v1 = m.pop_val(), v0 = m.pop_val(); /* second argument on top */
                        if (m.ok) m.vals.push_back(b.make(f, v0, v1, 0.f));
                    } else if (is_func(f) && m.ok) {
                        const int v = m.pop_val();
                        if (m.ok) m.vals.push_back(b.make(f, v, -1, 0.f));
                    }
                }
                break;
            case TOK_OP: m.ops.push_back(t.text[0]); break;
        }
        if (!m.ok) return false;
    }
    while (m.ok && !m.ops.empty()) m.reduce();
    if (!m.ok || m.vals.empty()) return false;
    e.root = m.vals.back(); /* the reference returns the top of the operand stack (evaluator.cpp:105) */
    return true;
}

static void postfix_rec(const Expr& e, int n, std::string& s) {
    const Node& nd = e.nodes[n];
    char buf[64];
    switch (nd.kind) {
        case 'x': case 'y': case 'z': s += nd.kind; break;
        case 'c': std::snprintf(buf, sizeof buf, "%g", (double)nd.value); s += buf; break;
        case 'N': postfix_rec(e, nd.a, s); s += " NEG"; return;
        case 'S': postfix_rec(e, nd.a, s); s += " sin"; return;
        case 'C': postfix_rec(e, nd.a, s); s += " cos"; return;
        case 'Q': postfix_rec(e, nd.a, s); s += " sqrt"; return;
        case 'A': postfix_rec(e, nd.a, s); s += " abs"; return;
        case 'm': case 'M': postfix_rec(e, nd.a, s); s += ' '; postfix_rec(e, nd.b, s); s += nd.kind == 'm' ? " min" : " max"; return;
        default: postfix_rec(e, nd.a, s); s += ' '; postfix_rec(e, nd.b, s); s += ' '; s += nd.kind; return;
    }
}
std::string postfix_text(const Expr& e) {
    std::string s;
    if (e.root >= 0) postfix_rec(e, e.root, s);
    return s;
}

/* ------------------------------------------------------------------------------------------------------------ */

namespace {

struct Lowerer {
    const Expr& e;
    Compiled& out;
    std::map<int, int> const_slot; /* node -> slot index */
    std::map<int, int> axis_slot;
    std::map<uint32_t, int> literal_index;
    bool overflow = false;
    Lowerer(const Expr& ex, Compiled& o) : e(ex), out(o) {}

    static bool leaf(const Node& n) { return n.kind == 'x' || n.kind == 'y' || n.kind == 'z' || n.kind == 'c'; }

    int literal(float v) {
        uint32_t bits;
        std::memcpy(&bits, &v, 4);
        auto it = literal_index.find(bits);
        if (it != literal_index.end()) return it->second;
        int idx = (int)out.kpool.size();
        out.kpool.push_back(v);
        literal_index[bits] = idx;
        return idx;
    }

    void collect_literals(int n, std::vector<char>& seen) {
        if (seen[n]) return;
        seen[n] = 1;
        const Node& nd = e.nodes[n];
        if (nd.kind == 'c') literal(nd.value);
        if (nd.a >= 0) collect_literals(nd.a, seen);
        if (nd.b >= 0) collect_literals(nd.b, seen);
    }

    /* maximal constant subtrees and maximal single-variable subtrees */
    void find_slots(int n, bool inside_axis) {
        const Node& nd = e.nodes[n];
        if (leaf(nd)) {
            /* a bare variable outside any hoisted subtree is the trivial one-variable subtree: the grid kernel then
             * reads the scaled coordinate from an axis table like every other per-axis value */
            if (nd.kind != 'c' && !inside_axis && !axis_slot.count(n)) { int s = (int)axis_slot.size(); axis_slot[n] = s; }
            return;
        }
        if (nd.mask == 0) {
            if (!const_slot.count(n)) { int s = (int)const_slot.size(); const_slot[n] = s; }
            return;
        }
        if (!inside_axis && (nd.mask == 1 || nd.mask == 2 || nd.mask == 4)) {
            if (!axis_slot.count(n)) { int s = (int)axis_slot.size(); axis_slot[n] = s; }
            inside_axis = true; /* keep descending only to find constant subtrees */
        }
        if (nd.a >= 0) find_slots(nd.a, inside_axis);
        if (nd.b >= 0) find_slots(nd.b, inside_axis);
    }

    enum Mode { POINT, GRID, LITERAL }; /* LITERAL: constant-slot programs, built from literals only */

    /* does `n` become a single push in this mode (when it is not the root of the program being generated)? */
    bool is_push(int n, Mode mode, int self) const {
        if (n == self) return leaf(e.nodes[n]);
        if (leaf(e.nodes[n])) return true;
        if (mode != LITERAL && const_slot.count(n)) return true;
        if (mode == GRID && axis_slot.count(n)) return true;
        return false;
    }
    int need(int n, Mode mode, int self, std::map<int, int>& memo) const {
        if (is_push(n, mode, self)) return 1;
        auto it = memo.find(n);
        if (it != memo.end()) return it->second;
        const Node& nd = e.nodes[n];
        int r;
        if (nd.b < 0) r = need(nd.a, mode, self, memo); /* 'N' and the functions */
        else {
            int l = need(nd.a, mode, self, memo), rr = need(nd.b, mode, self, memo);
            r = (l == rr) ? l + 1 : std::max(l, rr);
        }
        memo[n] = r;
        return r;
    }
    void gen(int n, Mode mode, int self, std::vector<uint32_t>& code, std::map<int, int>& memo) {
        const Node& nd = e.nodes[n];
        if (n != self || leaf(nd)) {
            if (mode == GRID) {
                auto as = axis_slot.find(n);
                if (as != axis_slot.end()) {
                    int op = nd.mask == 1 ? MCB_OP_PUSH_TX : nd.mask == 2 ? MCB_OP_PUSH_TY : MCB_OP_PUSH_TZ;
                    code.push_back(MCB_INSN(op, axis_local[as->second]));
                    return;
                }
            }
            if (nd.kind == 'x') { code.push_back(MCB_INSN(MCB_OP_PUSH_X, 0)); return; }
            if (nd.kind == 'y') { code.push_back(MCB_INSN(MCB_OP_PUSH_Y, 0)); return; }
            if (nd.kind == 'z') { code.push_back(MCB_INSN(MCB_OP_PUSH_Z, 0)); return; }
            if (nd.kind == 'c') { code.push_back(MCB_INSN(MCB_OP_PUSH_K, literal(nd.value))); return; }
            auto cs = const_slot.find(n);
            if (mode != LITERAL && cs != const_slot.end()) { code.push_back(MCB_INSN(MCB_OP_PUSH_K, out.n_literals + cs->second)); return; }
        }
        if (nd.b < 0) { /* 'N' and the functions */
            gen(nd.a, mode, self, code, memo);
            code.push_back(MCB_INSN(nd.kind == 'N' ? MCB_OP_NEG : nd.kind == 'S' ? MCB_OP_SIN : nd.kind == 'C' ? MCB_OP_COS
                                    : nd.kind == 'Q' ? MCB_OP_SQRT : MCB_OP_ABS, 0));
            return;
        }
        int la = need(nd.a, mode, self, memo), lb = need(nd.b, mode, self, memo);
        bool right_first = lb > la;
        int op;
        switch (nd.kind) {
            case '+': op = MCB_OP_ADD; break;
            case '*': op = MCB_OP_MUL; break;
            case '-': op = right_first ? MCB_OP_RSUB : MCB_OP_SUB; break;
            case '/': op = right_first ? MCB_OP_RDIV : MCB_OP_DIV; break;
            case 'm': op = MCB_OP_MIN; break; /* commutative bit for bit (mcb_minf): either order, no reversed form */
            case 'M': op = MCB_OP_MAX; break;
            default: op = right_first ? MCB_OP_RPOW : MCB_OP_POW; break;
        }
        if (right_first) { gen(nd.b, mode, self, code, memo); gen(nd.a, mode, self, code, memo); }
        else { gen(nd.a, mode, self, code, memo); gen(nd.b, mode, self, code, memo); }
        code.push_back(MCB_INSN(op, 0));
    }
    std::vector<int> axis_local; /* axis slot -> index within its own axis' table set */

    static int depth_of(const std::vector<uint32_t>& code, size_t b, size_t n) {
        int sp = 0, mx = 0;
        for (size_t i = b; i < b + n; i++) {
            uint32_t op = MCB_INSN_OP(code[i]);
            if (op >= MCB_OP_PUSH_X && op <= MCB_OP_PUSH_TZ) sp++;
            else if (!MCB_OP_IS_UNARY(op) && op != MCB_OP_END) sp--;
            mx = std::max(mx, sp);
        }
        return mx;
    }

    int run() {
        std::vector<char> seen(e.nodes.size(), 0);
        collect_literals(e.root, seen);
        out.n_literals = (int)out.kpool.size();
        find_slots(e.root, false);

        /* order: constant slots (by slot id), then axis slots */
        std::vector<int> cnode(const_slot.size()), anode(axis_slot.size());
        for (auto& kv : const_slot) cnode[kv.second] = kv.first;
        for (auto& kv : axis_slot) anode[kv.second] = kv.first;
        axis_local.assign(anode.size(), 0);
        for (size_t s = 0; s < anode.size(); s++) {
            int ax = e.nodes[anode[s]].mask == 1 ? 0 : e.nodes[anode[s]].mask == 2 ? 1 : 2;
            axis_local[s] = out.n_axis_slots[ax]++;
        }
        out.kpool.resize(out.n_literals + cnode.size(), 0.0f);

        for (size_t s = 0; s < cnode.size() + anode.size(); s++) {
            bool is_const = s < cnode.size();
            int node = is_const ? cnode[s] : anode[s - cnode.size()];
            Slot sl;
            sl.node = node;
            sl.axis = is_const ? -1 : (e.nodes[node].mask == 1 ? 0 : e.nodes[node].mask == 2 ? 1 : 2);
            sl.kindex = is_const ? out.n_literals + (int)s : axis_local[s - cnode.size()];
            sl.code_begin = (int)out.slot_code.size();
            std::map<int, int> memo;
            gen(node, is_const ? LITERAL : POINT, node, out.slot_code, memo);
            sl.code_len = (int)out.slot_code.size() - sl.code_begin;
            out.slot_depth = std::max(out.slot_depth, depth_of(out.slot_code, sl.code_begin, sl.code_len));
            out.slots.push_back(sl);
        }
        {
            std::map<int, int> memo;
            gen(e.root, POINT, -1, out.point_code, memo);
            out.point_depth = depth_of(out.point_code, 0, out.point_code.size());
        }
        {
            std::map<int, int> memo;
            gen(e.root, GRID, -1, out.grid_code, memo);
            out.grid_depth = depth_of(out.grid_code, 0, out.grid_code.size());
            out.grid_fused_depth = fuse(out.grid_code, out.grid_fused);
        }
        if (out.point_code.size() > MCB_MAX_CODE || out.grid_code.size() > MCB_MAX_CODE ||
            out.slot_code.size() > 4 * MCB_MAX_CODE || out.kpool.size() > MCB_MAX_K ||
            out.slots.size() > MCB_MAX_SLOTS || out.point_depth > MCB_MAX_STACK || out.slot_depth > MCB_MAX_STACK ||
            out.grid_depth > MCB_MAX_STACK)
            return MCB_E_CAPACITY;
        for (const Slot& sl : out.slots)
            if (sl.code_len > MCB_MAX_CODE) return MCB_E_CAPACITY;
        return MCB_OK;
    }
};

} /* namespace */

int compile(const std::string& eq, Compiled& out, std::string* err, int grammar) {
    out = Compiled();
    std::vector<Token> toks;
    if (!tokenize(eq, toks, &out.equation, grammar)) {
        if (err) *err = grammar == GRAMMAR_FUNCTIONS ? "parse error (function grammar: the reference's language plus sin( cos( sqrt( abs( min( max()"
                                                     : "parse error (Evaluator::tokenize rejects this equation)";
        return MCB_E_PARSE;
    }
    if (!build_expr(toks, out.expr)) {
        if (err) *err = "equation is accepted by the reference tokenizer but underflows its operand stack (undefined behaviour there); refused";
        return MCB_E_PARSE;
    }
    Lowerer lw(out.expr, out);
    int rc = lw.run();
    if (rc != MCB_OK && err) *err = "equation too large for the bytecode limits (MCB_MAX_CODE/MCB_MAX_K/MCB_MAX_SLOTS/MCB_MAX_STACK)";
    return rc;
}

/* Postfix -> fused accumulator form (mcb_bytecode.h).  A push directly followed by a binary operator becomes that
 * operator's operand; the other pushes keep spilling the accumulator, except the very first value of the program,
 * which is a plain load.  Returns the number of memory-stack levels the fused program needs. */
int fuse(const std::vector<uint32_t>& postfix, std::vector<uint32_t>& fused) {
    fused.clear();
    auto is_push = [](uint32_t op) { return op >= MCB_OP_PUSH_X && op <= MCB_OP_PUSH_TZ; };
    auto is_bin = [](uint32_t op) { return (op >= MCB_OP_ADD && op <= MCB_OP_RPOW) || op == MCB_OP_MIN || op == MCB_OP_MAX; };
    static const int direct[] = {MCB_F_ADD, MCB_F_SUB, MCB_F_RSUB, MCB_F_MUL, MCB_F_DIV, MCB_F_RDIV, MCB_F_POW, MCB_F_RPOW};
    static const int popped[] = {MCB_F_ADD, MCB_F_RSUB, MCB_F_SUB, MCB_F_MUL, MCB_F_RDIV, MCB_F_DIV, MCB_F_RPOW, MCB_F_POW};
    /* the fused word of binary operator op with operand src; min and max are one op, bit 3 of src picks max */
    auto bin_word = [](uint32_t op, bool pop, uint32_t src, uint32_t arg) -> uint32_t {
        if (op == MCB_OP_MIN || op == MCB_OP_MAX) return MCB_FINSN(MCB_F_MINMAX, src | (op == MCB_OP_MAX ? MCB_SRC_MAX_BIT : 0u), arg);
        return MCB_FINSN((pop ? popped : direct)[op - MCB_OP_ADD], src, arg);
    };
    int depth = 0, mem = 0, mem_max = 0; /* depth: values on the operand stack (accumulator included) */
    for (size_t i = 0; i < postfix.size(); i++) {
        const uint32_t w = postfix[i], op = MCB_INSN_OP(w), arg = MCB_INSN_ARG(w);
        if (op == MCB_OP_END) break;
        if (is_push(op)) {
            const uint32_t src = op - MCB_OP_PUSH_X; /* PUSH_X..PUSH_TZ map onto MCB_SRC_X..MCB_SRC_TZ in order */
            const uint32_t nop = i + 1 < postfix.size() ? MCB_INSN_OP(postfix[i + 1]) : (uint32_t)MCB_OP_END;
            if (depth >= 1 && is_bin(nop)) { /* acc = second, leaf = top */
                fused.push_back(bin_word(nop, false, src, arg));
                i++;
            } else if (depth == 0) {
                fused.push_back(MCB_FINSN(MCB_F_LOAD, src, arg));
                depth = 1;
            } else {
                fused.push_back(MCB_FINSN(MCB_F_PUSH, src, arg));
                depth++;
                mem_max = std::max(mem_max, ++mem);
            }
        } else if (op == MCB_OP_NEG) {
            fused.push_back(MCB_FINSN(MCB_F_NEG, 0, 0));
        } else if (op >= MCB_OP_SIN && op <= MCB_OP_ABS) {
            fused.push_back(MCB_FINSN(MCB_F_SIN + (op - MCB_OP_SIN), 0, 0));
        } else { /* binary operator on two stacked values: acc = top, popped = second */
            fused.push_back(bin_word(op, true, MCB_SRC_POP, 0));
            depth--;
            mem--;
        }
    }
    return mem_max;
}

std::string disassemble_fused(const std::vector<uint32_t>& code) {
    static const char* fops[] = {"LOAD", "PUSH", "ADD", "SUB", "RSUB", "MUL", "DIV", "RDIV", "POW", "RPOW", "NEG",
                                 "SIN", "COS", "SQRT", "ABS", "?", "MIN", "MAX"};
    static const char* srcs[] = {"X", "Y", "Z", "K", "TX", "TY", "TZ", "POP"};
    std::string s;
    char buf[48];
    for (uint32_t w : code) {
        uint32_t fop = MCB_FINSN_OP(w), src = MCB_FINSN_SRC(w);
        MCB_FINSN_DECODE(fop, src);
        if (!s.empty()) s += "; ";
        s += fops[fop];
        if (fop == MCB_F_NEG || MCB_F_IS_FN(fop)) continue;
        s += ' ';
        s += src <= MCB_SRC_POP ? srcs[src] : "?";
        if (src >= MCB_SRC_K && src <= MCB_SRC_TZ) {
            std::snprintf(buf, sizeof buf, "%u", MCB_FINSN_ARG(w));
            s += buf;
        }
    }
    return s;
}

std::string disassemble(const std::vector<uint32_t>& code) {
    static const char* names[] = {"END", "X", "Y", "Z", "K", "TX", "TY", "TZ", "ADD", "SUB", "RSUB",
                                  "MUL", "DIV", "RDIV", "POW", "RPOW", "NEG", "SIN", "COS", "SQRT", "ABS", "MIN", "MAX"};
    std::string s;
    char buf[32];
    for (uint32_t w : code) {
        uint32_t op = MCB_INSN_OP(w);
        if (!s.empty()) s += ' ';
        s += op < MCB_OP_COUNT ? names[op] : "?";
        if (op >= MCB_OP_PUSH_K && op <= MCB_OP_PUSH_TZ) {
            std::snprintf(buf, sizeof buf, "%u", MCB_INSN_ARG(w));
            s += buf;
        }
    }
    return s;
}

} /* namespace mcb */
