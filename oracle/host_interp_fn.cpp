/* TEST INFRASTRUCTURE ONLY — oracle/host_interp.cpp (compiled into this file unchanged) under a grammar chosen at run
 * time: every mcoh_* function lowers its equation with mcb::compile(..., grammar) instead of the reference grammar, so the
 * product's bytecode for function equations (mcb.h, MCB_GRAMMAR_FUNCTIONS) runs on the host in the CPU tier.
 *   void mcoh_set_grammar(int grammar)   MCB_GRAMMAR_REFERENCE (the default) or MCB_GRAMMAR_FUNCTIONS
 * Built by tests/functions_common.py with -ffp-contract=off, like oracle/Makefile builds host_interp.cpp. */
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "../marching-cube-for-implicit-surfaces_b200/csrc/mcb_lower.h"

static int g_grammar = mcb::GRAMMAR_REFERENCE;

/* host_interp.cpp calls mcb::compile(eq, c, nullptr): the three-argument calls take the grammar chosen above */
#define compile(eq, c, err) compile(eq, c, err, g_grammar)
#include "host_interp.cpp"
#undef compile

extern "C" void mcoh_set_grammar(int grammar) { g_grammar = grammar; }
