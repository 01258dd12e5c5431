/* Host-side front end of the evaluator: equation string -> tokens -> expression DAG -> bytecode programs.
 *
 * Semantics are the reference's, not a conventional parser's:
 *   - tokenizer:  Evaluator::tokenize, evaluator.cpp:139-237 (implicit '*', unary NEG, bracket balance, numbers)
 *   - evaluation: Evaluator::evaluate / evaluate_op, evaluator.cpp:22-107 — a two-stack walk that never reduces on
 *     push, reduces at ')' and at the end, and looks back ONE operator for precedence (evaluator.cpp:32-37).  Every
 *     chain of equal precedence therefore associates to the right, `-x^2` is (-x)^2, `x*-y+z` is x*(-y+z), ...
 * The control flow of that walk depends only on the token sequence, never on values, so we run it once
 * symbolically (operand stack of DAG node ids) and obtain the exact operation tree the reference executes per
 * point; emitting that tree as bytecode reproduces each fp32 operation with the same operands.
 *
 * The lowering then does the optimisations a compiler may do without changing a single bit of any result:
 *   - common sub-expressions share a node;
 *   - maximal constant subtrees are evaluated once (on the device, by the same interpreter) into the constant
 *     pool -> OP_PUSH_K;
 *   - maximal subtrees that depend on ONE variable only are evaluated once per grid coordinate into per-axis
 *     tables (loop-invariant code motion over the regular grid) -> OP_PUSH_TX/TY/TZ;
 *   - operand evaluation order is chosen Sethi-Ullman style (operands are pure, order cannot change values) with
 *     reversed opcodes keeping each operand in its role, so the register-cached operand stack stays shallow.
 */
#ifndef MCB_LOWER_H
#define MCB_LOWER_H

#include <cstdint>
#include <string>
#include <vector>

#include "mcb_bytecode.h"

namespace mcb {

enum TokType { TOK_OP, TOK_NUM, TOK_VAR, TOK_BRAC_O, TOK_BRAC_C, TOK_NEG, TOK_FUNC, TOK_COMMA };
struct Token {
    TokType type;
    std::string text; /* "NEG" for unary minus, like the reference; "sin(" etc. for a function and its bracket; "," */
};

/* Grammars (mcb.h): MCB_GRAMMAR_REFERENCE = the reference's language; MCB_GRAMMAR_FUNCTIONS adds sin( cos( sqrt( abs(
 * and the two-argument min( max(.  A function name and its '(' are one TOK_FUNC token that takes part in implicit
 * multiplication, the unary-minus rule and bracket balance exactly as '(' does; the walk applies the function at the
 * matching ')'.  Inside a min( / max( bracket exactly one ',' (TOK_COMMA) separates the two arguments: before it the rules
 * that precede ')' apply, after it those that follow '('; the walk reduces each argument down to the function's marker,
 * as ')' reduces a bracket, so `max(x-y+z,0)` is max(x-(y+z),0).  A ',' anywhere else is a parse error. */
enum { GRAMMAR_REFERENCE = 0, GRAMMAR_FUNCTIONS = 1 };

/* Evaluator::tokenize (evaluator.cpp:139-237). false = parse error. `cleaned` = equation with spaces removed. */
bool tokenize(const std::string& eq, std::vector<Token>& out, std::string* cleaned, int grammar = GRAMMAR_REFERENCE);

struct Node {
    char kind;  /* 'x','y','z' variable; 'c' literal; '+','-','*','/','^' binary (a op b); 'N' negate a;
                 * 'S' sin a, 'C' cos a, 'Q' sqrt a, 'A' abs a, 'm' min(a,b), 'M' max(a,b) (function grammar) */
    int a, b;   /* children (node ids), -1 when unused */
    float value; /* literal value (strtof, like stof at evaluator.cpp:82) */
    uint8_t mask; /* variables the subtree depends on: 1=x 2=y 4=z */
};

struct Expr {
    std::vector<Node> nodes;
    int root = -1;
};

/* Symbolic run of Evaluator::evaluate. false when the reference would underflow its operand stack (it accepts
 * e.g. "x+" and then reads outside its stack — undefined behaviour we refuse to guess at). */
bool build_expr(const std::vector<Token>& toks, Expr& e);

/* Postfix text in the reference's own evaluation order (left operand, right operand, operator), for tests:
 * "x-y+z" -> "x y z + -". */
std::string postfix_text(const Expr& e);

struct Slot {
    int node;       /* DAG node whose value the slot caches */
    int axis;       /* 0,1,2 = per-x/y/z table; -1 = folded constant (value -> constant pool) */
    int kindex;     /* constant-pool index for axis == -1 */
    int code_begin; /* its program inside Compiled::slot_code */
    int code_len;
};

struct Compiled {
    std::string equation; /* cleaned text */
    Expr expr;
    std::vector<uint32_t> point_code; /* full expression, arbitrary (x,y,z); uses PUSH_K but no tables */
    std::vector<uint32_t> grid_code;  /* full expression on the grid; uses PUSH_K and PUSH_T* */
    std::vector<uint32_t> grid_fused; /* grid_code in the fused accumulator form the grid kernel runs */
    int grid_fused_depth = 0;         /* memory-stack levels grid_fused needs */
    std::vector<uint32_t> slot_code;  /* programs of all slots, concatenated */
    std::vector<Slot> slots;          /* constant slots first, then axis slots */
    std::vector<float> kpool;         /* literals (exact strtof bits); folded slots are filled in by the device */
    int n_literals = 0;               /* kpool[0..n_literals) are literals, the rest folded constants */
    int n_axis_slots[3] = {0, 0, 0};
    int point_depth = 0, grid_depth = 0, slot_depth = 0; /* operand-stack depth each program needs */
};

/* tokenize + build + lower. Returns MCB_OK / MCB_E_PARSE / MCB_E_CAPACITY (program or pool too large). */
int compile(const std::string& eq, Compiled& out, std::string* err, int grammar = GRAMMAR_REFERENCE);

std::string disassemble(const std::vector<uint32_t>& code);

/* postfix words -> fused accumulator words (mcb_bytecode.h); returns the memory-stack depth of the result */
int fuse(const std::vector<uint32_t>& postfix, std::vector<uint32_t>& fused);
std::string disassemble_fused(const std::vector<uint32_t>& code);

} /* namespace mcb */

#endif
