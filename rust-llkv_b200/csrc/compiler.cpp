// compiler.cpp — see compiler.h.  Turns the reference's predicate program / scalar expressions / aggregate specs into
// the stack program of the fused scan kernel.  No CUDA here.
#include "compiler.h"

#include <algorithm>

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <stdexcept>

namespace llkv {

typedef __int128 i128;
typedef unsigned __int128 u128;

namespace {

struct CompileError {
  int32_t code;
  std::string msg;
};

[[noreturn]] void fail(int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  throw CompileError{code, buf};
}

// ---------------------------------------------------------------- DataType algebra (llkv-compute/src/kernels.rs:38-45,179-242)
struct DT {
  int type = LLKV_PT_NULL, p = 0, s = 0;
};
DT dt(int t, int p = 0, int s = 0) {
  DT d;
  d.type = t;
  d.p = p;
  d.s = s;
  return d;
}
bool dt_eq(DT a, DT b) { return a.type == b.type && (a.type != LLKV_PT_DECIMAL128 || (a.p == b.p && a.s == b.s)); }

enum Kind { K_NULL, K_I64, K_U64, K_F64, K_DEC, K_BOOL, K_DATE32, K_STR };

bool type_is_signed_int(int t) {
  return t == LLKV_PT_INT8 || t == LLKV_PT_INT16 || t == LLKV_PT_INT32 || t == LLKV_PT_INT64 || t == LLKV_PT_DATE32 ||
         t == LLKV_PT_DATE64;
}
bool type_is_unsigned_int(int t) {
  return t == LLKV_PT_UINT8 || t == LLKV_PT_UINT16 || t == LLKV_PT_UINT32 || t == LLKV_PT_UINT64;
}
int type_bits(int t) {
  switch (t) {
    case LLKV_PT_INT8: case LLKV_PT_UINT8: return 8;
    case LLKV_PT_INT16: case LLKV_PT_UINT16: return 16;
    case LLKV_PT_INT32: case LLKV_PT_UINT32: case LLKV_PT_DATE32: return 32;
    default: return 64;
  }
}
bool is_float_t(int t) { return t == LLKV_PT_FLOAT64 || t == LLKV_PT_FLOAT32; }
bool is_int_t(int t) {
  return (type_is_signed_int(t) && t != LLKV_PT_DATE32 && t != LLKV_PT_DATE64) || type_is_unsigned_int(t);
}
Kind kind_of_type(int t) {
  switch (t) {
    case LLKV_PT_NULL: return K_NULL;
    case LLKV_PT_FLOAT64: case LLKV_PT_FLOAT32: return K_F64;
    case LLKV_PT_DECIMAL128: return K_DEC;
    case LLKV_PT_BOOLEAN: return K_BOOL;
    case LLKV_PT_UTF8: return K_STR;
    case LLKV_PT_DATE32: return K_DATE32;
    default: return type_is_unsigned_int(t) ? K_U64 : K_I64;
  }
}
DT coerce_decimals(int lp, int ls, int rp, int rs) {
  const int scale = ls > rs ? ls : rs;
  const int li = lp - ls, ri = rp - rs;
  const int id = li > ri ? li : ri;
  int prec = id + scale;
  if (prec < 1) prec = 1;
  if (prec > 38) prec = 38;
  return dt(LLKV_PT_DECIMAL128, prec, scale);
}
DT common_type(DT l, DT r) {
  if (dt_eq(l, r)) return l;
  if (l.type == LLKV_PT_NULL) return r;
  if (r.type == LLKV_PT_NULL) return l;
  if (l.type == LLKV_PT_DECIMAL128 && r.type == LLKV_PT_DECIMAL128) return coerce_decimals(l.p, l.s, r.p, r.s);
  if (l.type == LLKV_PT_DECIMAL128 || r.type == LLKV_PT_DECIMAL128) {
    const DT d = l.type == LLKV_PT_DECIMAL128 ? l : r, o = l.type == LLKV_PT_DECIMAL128 ? r : l;
    if (is_float_t(o.type)) return dt(LLKV_PT_FLOAT64);
    if (is_int_t(o.type)) return coerce_decimals(d.p, d.s, 38, 0);
    return dt(LLKV_PT_FLOAT64);
  }
  if (is_float_t(l.type) || is_float_t(r.type)) return dt(LLKV_PT_FLOAT64);
  if (is_int_t(l.type) && is_int_t(r.type)) {
    const bool ls = type_is_signed_int(l.type), rs = type_is_signed_int(r.type);
    const int lb = type_bits(l.type), rb = type_bits(r.type);
    const int mx = lb > rb ? lb : rb;
    if (ls != rs) return mx >= 64 ? dt(LLKV_PT_FLOAT64) : dt(LLKV_PT_INT64);
    if (ls) return dt(mx >= 64 ? LLKV_PT_INT64 : mx >= 32 ? LLKV_PT_INT32 : mx >= 16 ? LLKV_PT_INT16 : LLKV_PT_INT8);
    return dt(mx >= 64 ? LLKV_PT_UINT64 : mx >= 32 ? LLKV_PT_UINT32 : mx >= 16 ? LLKV_PT_UINT16 : LLKV_PT_UINT8);
  }
  return dt(LLKV_PT_FLOAT64);
}

i128 lit_i128(const llkv_literal& l) { return (i128)(((u128)l.hi << 64) | (u128)l.lo); }
double lit_f64(const llkv_literal& l) {
  double d;
  memcpy(&d, &l.lo, 8);
  return d;
}
uint64_t f64_bits(double d) {
  uint64_t b;
  memcpy(&b, &d, 8);
  return b;
}
i128 pow10_i128(int k) {
  i128 v = 1;
  for (int i = 0; i < k; ++i) v *= 10;
  return v;
}
int digits_i128(i128 v) {
  u128 a = v < 0 ? (u128)0 - (u128)v : (u128)v;
  int d = 1;
  while (a >= 10) {
    a /= 10;
    ++d;
  }
  return d;
}
bool fits_i64(i128 v) { return v >= (i128)INT64_MIN && v <= (i128)INT64_MAX; }
i128 floor_div(i128 a, i128 b) {  // b > 0
  i128 q = a / b, r = a % b;
  if (r != 0 && a < 0) q -= 1;
  return q;
}
i128 ceil_div(i128 a, i128 b) {  // b > 0
  i128 q = a / b, r = a % b;
  if (r != 0 && a > 0) q += 1;
  return q;
}
bool pack_short_string(const uint8_t* p, uint32_t len, uint64_t* out) {
  if (len > 7) return false;
  uint64_t k = 0;
  for (uint32_t i = 0; i < len; ++i) k |= (uint64_t)p[i] << (56 - 8 * i);
  *out = k | len;
  return true;
}
DT literal_type(const llkv_literal& l) {  // eval.rs:166-186
  switch (l.kind) {
    case LLKV_LIT_BOOLEAN: return dt(LLKV_PT_BOOLEAN);
    case LLKV_LIT_INT128: return dt(LLKV_PT_INT64);
    case LLKV_LIT_FLOAT64: return dt(LLKV_PT_FLOAT64);
    case LLKV_LIT_DECIMAL128: return dt(LLKV_PT_DECIMAL128, digits_i128(lit_i128(l)), l.scale);
    case LLKV_LIT_DATE32: return dt(LLKV_PT_DATE32);
    case LLKV_LIT_STRING: return dt(LLKV_PT_UTF8);
    default: return dt(LLKV_PT_NULL);
  }
}

// arrow decimal result types of numeric::{add,sub,mul} on equal-typed operands
DT arith_type(DT l, DT r, int op) {
  if (kind_of_type(l.type) != K_DEC) return l;
  if (op == LLKV_BIN_ADD || op == LLKV_BIN_SUB) {
    const int s = l.s > r.s ? l.s : r.s;
    const int a = l.p - l.s > r.p - r.s ? l.p - l.s : r.p - r.s;
    const int p = a + s + 1;
    return dt(LLKV_PT_DECIMAL128, p > 38 ? 38 : p, s);
  }
  if (op == LLKV_BIN_MUL) {
    if (l.s + r.s > 38) fail(LLKV_ERR_INTERNAL, "Invalid argument error: Output scale of mul exceeds 38");
    const int p = l.p + r.p + 1;
    return dt(LLKV_PT_DECIMAL128, p > 38 ? 38 : p, l.s + r.s);
  }
  fail(LLKV_ERR_INTERNAL, "Decimal128 div/rem is not supported on this path");
}

// which casts the arrow-cast restatement covers (anything else: the reference's `cast(..).unwrap_or(array)` keeps the input)
bool cast_supported(DT from, DT to) {
  if (dt_eq(from, to)) return true;
  const Kind ik = kind_of_type(from.type), ok = kind_of_type(to.type);
  if (ik == K_NULL) return true;
  if ((ik == K_I64 || ik == K_DATE32) && ok == K_DEC) return true;
  if (ik == K_U64 && ok == K_DEC) return true;
  if (ik == K_DEC && ok == K_DEC) return true;
  if (ik == K_DEC && ok == K_F64) return true;
  if ((ik == K_I64 || ik == K_DATE32) && ok == K_F64) return true;
  if (ik == K_U64 && ok == K_F64) return true;
  if (ik == K_F64 && ok == K_I64) return true;
  if ((ik == K_I64 || ik == K_DATE32) && ok == K_I64) return true;
  if (ik == K_U64 && ok == K_I64) return true;
  if (ik == K_I64 && ok == K_U64) return true;
  if (ik == K_BOOL && ok == K_I64) return true;
  if (ik == K_I64 && ok == K_BOOL) return true;
  if (ik == K_F64 && ok == K_F64) return true;
  return false;
}

struct PNode {  // predicate tree rebuilt from the postfix program
  int op_index = -1;
  int tag = 0;
  std::vector<int> children;
};

struct VecInfo {
  DT t;
  bool scalar = false;
};

// ---------------------------------------------------------------- emitter
class Emitter {
 public:
  Emitter(const CompileRequest& req, CompileResult& out) : req_(req), out_(out) {
    col_plan_index_.assign(req.cols.size(), -1);
  }

  void run() {
    Plan& p = out_.plan;
    memset(&p, 0, sizeof(p));
    wide_ = req_.force_wide;
    // decimal columns with values beyond i64 can only run on the 128-bit interpreter: decided lazily in use_col()
    emit_selection();
    if (req_.bitmap_mode) {
      emit(OP_EMIT_BITMAP, 0, 0, 0);
      p.bitmap_mode = 1;
    } else {
      emit_keys();
      emit_aggregates();
    }
    emit(OP_END, 0, 0, 0);
    mark_filter_exits();
    finish();
  }

 private:
  const CompileRequest& req_;
  CompileResult& out_;
  std::vector<Instr> code_;
  std::vector<Lit> lits_;
  std::vector<int> col_plan_index_;
  std::vector<const ColumnMeta*> plan_cols_;
  std::vector<bool> nullable_;  // static "may be NULL" per stack entry
  int max_sp_ = 0;
  bool wide_ = false;
  bool can_narrow_fail_ = false;
  size_t select_end_ = 0;
  // expression nodes currently being compiled
  const llkv_scalar_node* nodes_ = nullptr;
  int n_nodes_ = 0;
  // accumulator words
  std::vector<uint8_t> gclass_;
  std::vector<FastWord> fast_;
  std::map<std::string, int> facts_;

  int sp() const { return (int)nullable_.size(); }

  // ---- low-level emission
  void emit(uint16_t op, uint8_t a, uint8_t b, uint32_t c) {
    if (code_.size() + 1 >= (size_t)kMaxInstr) fail(LLKV_ERR_INVALID_ARGUMENT, "query too large for one fused pass (%d instructions)", kMaxInstr);
    Instr in;
    in.op = op;
    in.a = a;
    in.b = b;
    in.c = c;
    code_.push_back(in);
  }
  void pushed(bool nullable) {
    nullable_.push_back(nullable);
    if (sp() > max_sp_) max_sp_ = sp();
    if (sp() > kMaxStackDepth) fail(LLKV_ERR_INVALID_ARGUMENT, "expression too deep for one fused pass (stack %d)", kMaxStackDepth);
  }
  void popped() { nullable_.pop_back(); }
  void set_top_nullable(bool v) { nullable_.back() = v; }
  bool get_top_nullable() const { return nullable_.back(); }

  uint32_t add_lit(uint64_t lo, uint64_t hi) {
    for (size_t i = 0; i < lits_.size(); ++i)
      if (lits_[i].lo == lo && lits_[i].hi == hi) return (uint32_t)i;
    if (lits_.size() >= (size_t)kMaxLits) fail(LLKV_ERR_INVALID_ARGUMENT, "too many literals for one fused pass (%d)", kMaxLits);
    Lit L;
    L.lo = lo;
    L.hi = hi;
    lits_.push_back(L);
    return (uint32_t)(lits_.size() - 1);
  }
  uint32_t add_lit_run(const std::vector<Lit>& run) {  // consecutive literals (ranges, IN lists)
    if (lits_.size() + run.size() > (size_t)kMaxLits) fail(LLKV_ERR_INVALID_ARGUMENT, "too many literals for one fused pass (%d)", kMaxLits);
    const uint32_t first = (uint32_t)lits_.size();
    for (const Lit& l : run) lits_.push_back(l);
    return first;
  }
  static Lit mk_lit_i(i128 v) {
    Lit L;
    L.lo = (uint64_t)(u128)v;
    L.hi = (uint64_t)((u128)v >> 64);
    return L;
  }
  void need_wide_for(i128 v) {
    if (!fits_i64(v)) wide_ = true;
  }

  int find_col(uint64_t fid) const {
    for (size_t i = 0; i < req_.cols.size(); ++i)
      if (req_.cols[i].field_id == fid) return (int)i;
    return -1;
  }
  int use_col(int ci) {
    if (col_plan_index_[ci] < 0) {
      if (plan_cols_.size() >= (size_t)kMaxCols) fail(LLKV_ERR_INVALID_ARGUMENT, "too many columns for one fused pass (%d)", kMaxCols);
      col_plan_index_[ci] = (int)plan_cols_.size();
      plan_cols_.push_back(&req_.cols[ci]);
      const ColumnMeta& c = req_.cols[ci];
      if (c.load_kind == LK_D128) {
        if (!c.dec_fits_i64) wide_ = true;
        can_narrow_fail_ = true;
      }
    }
    return col_plan_index_[ci];
  }
  void push_col(int ci) {
    const ColumnMeta& c = req_.cols[ci];
    emit(OP_PUSH_COL, (uint8_t)use_col(ci), c.load_kind, 0);
    pushed(c.nullable);
  }
  void push_lit_i(i128 v) {
    need_wide_for(v);
    const Lit L = mk_lit_i(v);
    emit(OP_PUSH_LIT, 0, 0, add_lit(L.lo, L.hi));
    pushed(false);
  }
  void push_lit_bits(uint64_t bits) {  // f64 bits / unsigned / packed string: hi = 0 keeps wide-mode reads of the low half exact
    emit(OP_PUSH_LIT, 0, 0, add_lit(bits, 0));
    pushed(false);
  }
  void push_null() {
    emit(OP_PUSH_LIT, 0, 1, add_lit(0, 0));
    pushed(true);
  }
  void binary(uint16_t op, uint8_t a, uint8_t b, bool result_nullable) {
    emit(op, a, b, 0);
    popped();
    popped();
    pushed(result_nullable);
  }

  // ---- selection phase: predicate program + MVCC ------------------------------------------------------------
  std::vector<PNode> ptree_;

  int build_tree(const ProgramView& pg) {
    std::vector<int> st;
    for (int i = 0; i < pg.n_ops; ++i) {
      const llkv_eval_op& op = pg.ops[i];
      PNode n;
      n.op_index = i;
      n.tag = op.tag;
      switch (op.tag) {
        case LLKV_EV_PUSH_PREDICATE: case LLKV_EV_PUSH_COMPARE: case LLKV_EV_PUSH_IN_LIST: case LLKV_EV_PUSH_IS_NULL:
        case LLKV_EV_PUSH_LITERAL:
          break;
        case LLKV_EV_FUSED_AND:
          if (op.child_count <= 0 || i + op.child_count > pg.n_ops - 1) fail(LLKV_ERR_INTERNAL, "FusedAnd runs past the end of the program");
          for (int k = 0; k < op.child_count; ++k)
            if (pg.ops[i + 1 + k].tag != LLKV_EV_FILTER_ITEM) fail(LLKV_ERR_INTERNAL, "FusedAnd expects filter items");
          i += op.child_count;
          break;
        case LLKV_EV_AND: case LLKV_EV_OR: {
          if (op.child_count <= 0 || (int)st.size() < op.child_count)
            fail(LLKV_ERR_INTERNAL, "%s opcode underflow", op.tag == LLKV_EV_AND ? "AND" : "OR");
          n.children.assign(st.end() - op.child_count, st.end());
          st.resize(st.size() - (size_t)op.child_count);
          break;
        }
        case LLKV_EV_NOT:
          if (st.empty()) fail(LLKV_ERR_INTERNAL, "NOT opcode underflow");
          n.children.push_back(st.back());
          st.pop_back();
          break;
        default: fail(LLKV_ERR_INTERNAL, "unknown eval op tag %d", op.tag);
      }
      ptree_.push_back(n);
      st.push_back((int)ptree_.size() - 1);
    }
    if (st.size() != 1) fail(LLKV_ERR_INTERNAL, "Program stack empty after evaluation");
    return st[0];
  }

  void emit_selection() {
    const ProgramView* pg = req_.prog;
    if (pg && pg->n_ops > 0) {
      nodes_ = pg->nodes;
      n_nodes_ = pg->n_nodes;
      const int root = build_tree(*pg);
      emit_top(root);
    }
    if (req_.mvcc.enabled && req_.mvcc.created_by && req_.mvcc.deleted_by) {
      const int cc = find_col(req_.mvcc.created_by->field_id), dc = find_col(req_.mvcc.deleted_by->field_id);
      if (cc < 0 || dc < 0) fail(LLKV_ERR_INTERNAL, "MVCC columns are not part of the table");
      if (req_.cols[cc].type != LLKV_PT_UINT64 || req_.cols[dc].type != LLKV_PT_UINT64)
        fail(LLKV_ERR_INVALID_ARGUMENT, "MVCC columns must be UInt64");
      if (req_.mvcc.noncommitted.size() > (size_t)kMaxNoncommitted)
        fail(LLKV_ERR_INVALID_ARGUMENT, "more than %d non-committed transactions in one snapshot", kMaxNoncommitted);
      emit(OP_MVCC, (uint8_t)use_col(cc), (uint8_t)use_col(dc), 0);
    }
    emit(OP_SELECT_DONE, 0, 0, 0);
    select_end_ = code_.size();
  }

  // top level: AND children become independent filters (only the rows bit matters at the root)
  void emit_top(int ni) {
    const PNode& n = ptree_[ni];
    const ProgramView& pg = *req_.prog;
    if (n.tag == LLKV_EV_AND) {
      for (int c : n.children) emit_top(c);
      return;
    }
    if (n.tag == LLKV_EV_FUSED_AND) {
      const llkv_eval_op& op = pg.ops[n.op_index];
      for (int k = 0; k < op.child_count; ++k) {
        emit_leaf(pg.ops[n.op_index + 1 + k]);
        emit(OP_FILTER, 0, 0, 0);
        popped();
      }
      return;
    }
    emit_pred(ni);
    emit(OP_FILTER, 0, 0, 0);
    popped();
  }

  void emit_pred(int ni) {
    const PNode& n = ptree_[ni];
    const ProgramView& pg = *req_.prog;
    const llkv_eval_op& op = pg.ops[n.op_index];
    switch (n.tag) {
      case LLKV_EV_PUSH_PREDICATE: emit_leaf(op); break;
      case LLKV_EV_FUSED_AND:
        for (int k = 0; k < op.child_count; ++k) {
          emit_leaf(pg.ops[n.op_index + 1 + k]);
          if (k) binary(OP_AND, 0, 0, true);
        }
        break;
      case LLKV_EV_PUSH_COMPARE: emit_compare_leaf(op.expr_left, op.cmp_op, op.expr_right); break;
      case LLKV_EV_PUSH_IN_LIST: emit_in_list_leaf(op); break;
      case LLKV_EV_PUSH_IS_NULL:
        check_node(op.expr_left);
        emit_batch_arrow(op.expr_left);
        emit(OP_ISNULL, (uint8_t)(op.negated != 0), 0, 0);
        set_top_nullable(false);
        break;
      case LLKV_EV_PUSH_LITERAL:
        emit(OP_BOOL_LIT, (uint8_t)(op.literal_bool != 0), 0, 0);
        pushed(false);
        break;
      case LLKV_EV_AND: case LLKV_EV_OR:
        for (size_t k = 0; k < n.children.size(); ++k) {
          emit_pred(n.children[k]);
          if (k) binary(n.tag == LLKV_EV_AND ? OP_AND : OP_OR, 0, 0, true);
        }
        break;
      case LLKV_EV_NOT:
        emit_pred(n.children[0]);
        emit(OP_NOT, 0, 0, 0);
        break;
      default: fail(LLKV_ERR_INTERNAL, "unknown eval op tag %d", n.tag);
    }
  }

  // typed predicate leaf: Filter{field, op} (typed_predicate.rs:252-315; literal casts literal.rs:368-519)
  void emit_leaf(const llkv_eval_op& op) {
    const ProgramView& pg = *req_.prog;
    const int ci = find_col(op.field_id);
    if (ci < 0) fail(LLKV_ERR_NOT_FOUND, "unknown field %llu", (unsigned long long)op.field_id);
    const ColumnMeta& c = req_.cols[ci];
    if (op.lit_begin < 0 || op.lit_count < 0 || op.lit_begin + op.lit_count > pg.n_literals)
      fail(LLKV_ERR_INTERNAL, "predicate literals out of range");
    const llkv_literal* l = pg.literals + op.lit_begin;
    push_col(ci);
    if (op.operator_tag == LLKV_OP_IS_NOT_NULL) { emit(OP_PRED_NOTNULL, 0, 0, 0); return; }
    if (op.operator_tag == LLKV_OP_IS_NULL) { emit(OP_PRED_ISNULL, 0, 0, 0); return; }
    if (op.operator_tag == LLKV_OP_RANGE && op.lower_kind == LLKV_BOUND_UNBOUNDED && op.upper_kind == LLKV_BOUND_UNBOUNDED) {
      emit(OP_PRED_ALL, 0, 0, 0);
      return;
    }
    if (c.dict_sorted) {
      emit_dict_leaf(c, op, l);
      return;
    }
    int lower = LLKV_BOUND_UNBOUNDED, upper = LLKV_BOUND_UNBOUNDED, eq = 0;
    const llkv_literal *ll = nullptr, *ul = nullptr;
    switch (op.operator_tag) {
      case LLKV_OP_EQUALS: case LLKV_OP_GT: case LLKV_OP_GTE: case LLKV_OP_LT: case LLKV_OP_LTE:
        if (op.lit_count != 1) fail(LLKV_ERR_INTERNAL, "operator needs one literal");
        if (op.operator_tag == LLKV_OP_EQUALS) { eq = 1; ll = l; }
        else if (op.operator_tag == LLKV_OP_GT) { lower = LLKV_BOUND_EXCLUDED; ll = l; }
        else if (op.operator_tag == LLKV_OP_GTE) { lower = LLKV_BOUND_INCLUDED; ll = l; }
        else if (op.operator_tag == LLKV_OP_LT) { upper = LLKV_BOUND_EXCLUDED; ul = l; }
        else { upper = LLKV_BOUND_INCLUDED; ul = l; }
        break;
      case LLKV_OP_RANGE: {
        int k = 0;
        lower = op.lower_kind;
        upper = op.upper_kind;
        if (lower != LLKV_BOUND_UNBOUNDED) ll = l + k++;
        if (upper != LLKV_BOUND_UNBOUNDED) ul = l + k++;
        if (k > op.lit_count) fail(LLKV_ERR_INTERNAL, "range bounds without literals");
        break;
      }
      case LLKV_OP_IN: emit_in_leaf(c, l, op.lit_count); return;
      case LLKV_OP_STARTS_WITH: case LLKV_OP_ENDS_WITH: case LLKV_OP_CONTAINS:
        if (op.lit_count != 1) fail(LLKV_ERR_INTERNAL, "operator needs one literal");
        emit_pattern_leaf(c, op.operator_tag, *l, op.literal_bool != 0);
        return;
      default: fail(LLKV_ERR_PREDICATE_BUILD, "operator lacks typed literal support");
    }
    // convert the bound literals to the column's native domain
    const int dom = col_domain(c);
    Lit a = {0, 0}, b = {0, 0};
    uint16_t opc = OP_PRED_I;
    if (dom == DOM_DEC) {
      opc = OP_PRED_D;
      // align literals and column to one scale; bounds are moved to the column's scale with exact floor/ceil
      int ds = c.scale;
      if (ll && ll->kind == LLKV_LIT_DECIMAL128 && ll->scale > ds) ds = ll->scale;
      if (ul && ul->kind == LLKV_LIT_DECIMAL128 && ul->scale > ds) ds = ul->scale;
      const i128 f = pow10_i128(ds - c.scale);
      if (eq) {
        const i128 r = dec_literal(*ll, ds);
        if (r % f != 0) {  // can never be equal: an empty range
          eq = 0;
          lower = LLKV_BOUND_EXCLUDED;
          a = mk_lit_i(~((i128)1 << 127));
          wide_ = true;
        } else {
          a = mk_lit_i(r / f);
          need_wide_for(r / f);
        }
      } else {
        if (ll) {
          const i128 r = dec_literal(*ll, ds);
          const i128 v = lower == LLKV_BOUND_INCLUDED ? ceil_div(r, f) : floor_div(r, f);
          a = mk_lit_i(v);
          need_wide_for(v);
        }
        if (ul) {
          const i128 r = dec_literal(*ul, ds);
          const i128 v = upper == LLKV_BOUND_INCLUDED ? floor_div(r, f) : ceil_div(r, f);
          (ll ? b : a) = mk_lit_i(v);
          need_wide_for(v);
        }
      }
    } else {
      opc = dom == DOM_I64 ? OP_PRED_I : (dom == DOM_F64 || dom == DOM_F32) ? OP_PRED_F : OP_PRED_U;
      if (ll) a = native_literal(c, dom, *ll);
      if (ul) (ll ? b : a) = native_literal(c, dom, *ul);
    }
    std::vector<Lit> run;
    run.push_back(a);
    if (ll && ul) run.push_back(b);
    const uint32_t first = add_lit_run(run);
    emit(opc, (uint8_t)(lower | (upper << 2) | (eq << 4)), 0, first);
  }

  enum { DOM_I64, DOM_U64, DOM_F64, DOM_F32, DOM_DEC, DOM_STR, DOM_BOOL };
  static int col_domain(const ColumnMeta& c) {
    if (c.type == LLKV_PT_FLOAT64) return DOM_F64;
    if (c.type == LLKV_PT_FLOAT32) return DOM_F32;
    if (c.type == LLKV_PT_DECIMAL128) return DOM_DEC;
    if (c.type == LLKV_PT_UTF8) return DOM_STR;
    if (c.type == LLKV_PT_BOOLEAN) return DOM_BOOL;
    if (type_is_unsigned_int(c.type)) return DOM_U64;
    return DOM_I64;
  }
  // decimal literal rescaled to `target` scale (>= its own)
  static i128 dec_literal(const llkv_literal& l, int target) {
    i128 raw;
    int ls;
    if (l.kind == LLKV_LIT_INT128) { raw = lit_i128(l); ls = 0; }
    else if (l.kind == LLKV_LIT_DECIMAL128) { raw = lit_i128(l); ls = l.scale; }
    else fail(LLKV_ERR_PREDICATE_BUILD, "literal type mismatch: expected decimal");
    i128 r;
    if (target < ls || __builtin_mul_overflow(raw, pow10_i128(target - ls), &r)) fail(LLKV_ERR_PREDICATE_BUILD, "decimal literal overflow");
    return r;
  }
  // FromLiteral for integer / float / bool / string natives
  Lit native_literal(const ColumnMeta& c, int dom, const llkv_literal& l) {
    Lit out = {0, 0};
    switch (dom) {
      case DOM_I64: case DOM_U64: {
        i128 v;
        if (l.kind == LLKV_LIT_INT128) v = lit_i128(l);
        else if (l.kind == LLKV_LIT_DECIMAL128 && l.scale == 0) v = lit_i128(l);
        else if (l.kind == LLKV_LIT_DATE32 && c.type == LLKV_PT_DATE32) v = (int64_t)l.lo;  // extension D4 (SURVEY.md §8a)
        else fail(LLKV_ERR_PREDICATE_BUILD, "literal type mismatch: expected integer");
        const int bits = type_bits(c.type);
        if (dom == DOM_I64) {
          const i128 lo = -((i128)1 << (bits - 1)), hi = ((i128)1 << (bits - 1)) - 1;
          if (v < lo || v > hi) fail(LLKV_ERR_PREDICATE_BUILD, "literal out of range for %d-bit integer", bits);
          out = mk_lit_i(v);
        } else {
          const i128 hi = bits == 64 ? (i128)UINT64_MAX : (((i128)1 << bits) - 1);
          if (v < 0 || v > hi) fail(LLKV_ERR_PREDICATE_BUILD, "literal out of range for unsigned %d-bit", bits);
          out.lo = (uint64_t)v;
        }
        return out;
      }
      case DOM_F64: case DOM_F32: {
        double v;
        if (l.kind == LLKV_LIT_FLOAT64) v = lit_f64(l);
        else if (l.kind == LLKV_LIT_INT128) v = (double)lit_i128(l);
        else if (l.kind == LLKV_LIT_DECIMAL128) {
          const i128 raw = lit_i128(l);
          v = raw == 0 ? 0.0 : (double)raw / powi_f64(10.0, l.scale);
        } else fail(LLKV_ERR_PREDICATE_BUILD, "literal type mismatch: expected float");
        if (dom == DOM_F32) {
          const float f = (float)v;
          if (!isfinite(f)) fail(LLKV_ERR_PREDICATE_BUILD, "float literal out of range for f32");
          v = (double)f;
        }
        out.lo = f64_bits(v);
        return out;
      }
      case DOM_BOOL:
        if (l.kind == LLKV_LIT_BOOLEAN) out.lo = l.lo != 0;
        else if (l.kind == LLKV_LIT_INT128 && (lit_i128(l) == 0 || lit_i128(l) == 1)) out.lo = (uint64_t)lit_i128(l);
        else fail(LLKV_ERR_PREDICATE_BUILD, "literal type mismatch: expected boolean");
        return out;
      case DOM_STR: {
        if (l.kind != LLKV_LIT_STRING) fail(LLKV_ERR_PREDICATE_BUILD, "literal type mismatch: expected string");
        const char* bytes;
        size_t len;
        literal_bytes(l, &bytes, &len);
        uint64_t packed = 0;
        if (!pack_short_string((const uint8_t*)bytes, (uint32_t)std::min<size_t>(len, 8), &packed))
          fail(LLKV_ERR_PREDICATE_BUILD, "string literal longer than 7 bytes against a short-string column");
        out.lo = packed;
        return out;
      }
    }
    fail(LLKV_ERR_INTERNAL, "bad domain");
  }

  // Typed leaves over a dictionary-coded Utf8 column (strings longer than 7 bytes): the resident values are ranks in the
  // byte-ordered dictionary, so every leaf becomes an integer leaf over ranks — equality and IN by looking the literal up,
  // ranges by lower/upper bound, patterns by testing each entry once here (typed_predicate.rs:75-209 on String).
  static std::string lit_string(const llkv_literal& l) {
    if (l.kind != LLKV_LIT_STRING) fail(LLKV_ERR_PREDICATE_BUILD, "literal type mismatch: expected string");
    const char* bytes;
    size_t len;
    literal_bytes(l, &bytes, &len);
    return std::string(bytes, len);
  }
  void emit_rank_range(int64_t lo, int64_t hi) {  // inclusive; lo > hi: nothing matches
    if (lo > hi) {
      emit(OP_IN_BITS, 0, 0, 0);
      return;
    }
    std::vector<Lit> run(2);
    run[0].lo = (uint64_t)lo; run[0].hi = 0;
    run[1].lo = (uint64_t)hi; run[1].hi = 0;
    emit(OP_PRED_U, (uint8_t)(LLKV_BOUND_INCLUDED | (LLKV_BOUND_INCLUDED << 2)), 0, add_lit_run(run));
  }
  void emit_rank_set(const std::vector<uint32_t>& ranks) {  // ascending
    if (ranks.empty()) { emit(OP_IN_BITS, 0, 0, 0); return; }
    if ((size_t)(ranks.back() - ranks.front()) + 1 == ranks.size()) { emit_rank_range(ranks.front(), ranks.back()); return; }
    if (ranks.size() > 255) fail(LLKV_ERR_PREDICATE_BUILD, "the predicate matches %zu scattered dictionary entries (at most 255 on this path)", ranks.size());
    std::vector<Lit> run(ranks.size());
    for (size_t i = 0; i < ranks.size(); ++i) { run[i].lo = ranks[i]; run[i].hi = 0; }
    emit(OP_IN_BITS, 0, (uint8_t)run.size(), add_lit_run(run));
  }
  void emit_dict_leaf(const ColumnMeta& c, const llkv_eval_op& op, const llkv_literal* l) {
    const std::vector<std::string>& dict = *c.dict_sorted;
    const int64_t D = (int64_t)dict.size();
    auto lb = [&](const std::string& x) { return (int64_t)(std::lower_bound(dict.begin(), dict.end(), x) - dict.begin()); };
    auto ub = [&](const std::string& x) { return (int64_t)(std::upper_bound(dict.begin(), dict.end(), x) - dict.begin()); };
    switch (op.operator_tag) {
      case LLKV_OP_EQUALS: case LLKV_OP_GT: case LLKV_OP_GTE: case LLKV_OP_LT: case LLKV_OP_LTE: {
        if (op.lit_count != 1) fail(LLKV_ERR_INTERNAL, "operator needs one literal");
        const std::string x = lit_string(l[0]);
        if (op.operator_tag == LLKV_OP_EQUALS) emit_rank_range(lb(x), ub(x) - 1);
        else if (op.operator_tag == LLKV_OP_GT) emit_rank_range(ub(x), D - 1);
        else if (op.operator_tag == LLKV_OP_GTE) emit_rank_range(lb(x), D - 1);
        else if (op.operator_tag == LLKV_OP_LT) emit_rank_range(0, lb(x) - 1);
        else emit_rank_range(0, ub(x) - 1);
        return;
      }
      case LLKV_OP_RANGE: {
        int k = 0;
        int64_t lo = 0, hi = D - 1;
        if (op.lower_kind != LLKV_BOUND_UNBOUNDED) {
          if (k >= op.lit_count) fail(LLKV_ERR_INTERNAL, "range bounds without literals");
          const std::string x = lit_string(l[k++]);
          lo = op.lower_kind == LLKV_BOUND_INCLUDED ? lb(x) : ub(x);
        }
        if (op.upper_kind != LLKV_BOUND_UNBOUNDED) {
          if (k >= op.lit_count) fail(LLKV_ERR_INTERNAL, "range bounds without literals");
          const std::string x = lit_string(l[k++]);
          hi = op.upper_kind == LLKV_BOUND_INCLUDED ? ub(x) - 1 : lb(x) - 1;
        }
        emit_rank_range(lo, hi);
        return;
      }
      case LLKV_OP_IN: {
        std::vector<uint32_t> ranks;
        for (int i = 0; i < op.lit_count; ++i) {
          const std::string x = lit_string(l[i]);
          const int64_t r = lb(x);
          if (r < D && dict[(size_t)r] == x) ranks.push_back((uint32_t)r);
        }
        std::sort(ranks.begin(), ranks.end());
        ranks.erase(std::unique(ranks.begin(), ranks.end()), ranks.end());
        emit_rank_set(ranks);
        return;
      }
      case LLKV_OP_STARTS_WITH: case LLKV_OP_ENDS_WITH: case LLKV_OP_CONTAINS: {
        if (op.lit_count != 1) fail(LLKV_ERR_INTERNAL, "operator needs one literal");
        std::string pat = lit_string(l[0]);
        const bool ci = op.literal_bool != 0;
        auto lower = [](std::string& x) { for (char& ch : x) if (ch >= 'A' && ch <= 'Z') ch = (char)(ch + 32); };
        if (ci) {
          for (char ch : pat) if ((unsigned char)ch >= 0x80) fail(LLKV_ERR_PREDICATE_BUILD, "case-insensitive patterns are ASCII-only on this path");
          if (c.str_non_ascii) fail(LLKV_ERR_PREDICATE_BUILD, "case-insensitive match over a column with non-ASCII strings is not on this path");
          lower(pat);
        }
        std::vector<uint32_t> ranks;
        for (int64_t r = 0; r < D; ++r) {
          std::string v = dict[(size_t)r];
          if (ci) lower(v);
          bool m;
          if (pat.size() > v.size()) m = false;
          else if (op.operator_tag == LLKV_OP_STARTS_WITH) m = v.compare(0, pat.size(), pat) == 0;
          else if (op.operator_tag == LLKV_OP_ENDS_WITH) m = v.compare(v.size() - pat.size(), pat.size(), pat) == 0;
          else m = v.find(pat) != std::string::npos;
          if (m) ranks.push_back((uint32_t)r);
        }
        emit_rank_set(ranks);
        return;
      }
      default: fail(LLKV_ERR_PREDICATE_BUILD, "operator lacks typed literal support");
    }
  }

  // StartsWith / EndsWith / Contains (typed_predicate.rs:187-209; only String implements them: :25-36 is `false` for every
  // other native type) over the packed short strings of this path.
  void emit_pattern_leaf(const ColumnMeta& c, int tag, const llkv_literal& l, bool ci) {
    if (col_domain(c) != DOM_STR) {  // the default trait methods: never matches; the domain stays the present rows
      emit(OP_IN_BITS, 0, 0, 0);
      return;
    }
    if (l.kind != LLKV_LIT_STRING) fail(LLKV_ERR_PREDICATE_BUILD, "literal type mismatch: expected string");
    const char* src;
    size_t full_len;
    literal_bytes(l, &src, &full_len);
    if (ci)
      for (size_t i = 0; i < full_len; ++i)
        if ((unsigned char)src[i] >= 0x80) fail(LLKV_ERR_PREDICATE_BUILD, "case-insensitive patterns are ASCII-only on this path");
    uint8_t bytes[16] = {0};
    memcpy(bytes, src, std::min<size_t>(full_len, 16));
    const uint32_t len = (uint32_t)std::min<size_t>(full_len, 16);  // (anything above 7 matches no short string)
    if (ci) {
      // to_lowercase() is Unicode's: ASCII lowering equals it exactly when neither side holds a non-ASCII character
      for (uint32_t i = 0; i < len; ++i) {
        if (bytes[i] >= 0x80) fail(LLKV_ERR_PREDICATE_BUILD, "case-insensitive patterns are ASCII-only on this path");
        if (bytes[i] >= 'A' && bytes[i] <= 'Z') bytes[i] = (uint8_t)(bytes[i] + 32);
      }
      if (c.str_non_ascii) fail(LLKV_ERR_PREDICATE_BUILD, "case-insensitive match over a column with non-ASCII strings is not on this path");
    }
    if (len > 7) {  // no string of a short-string column is that long
      emit(OP_IN_BITS, 0, 0, 0);
      return;
    }
    uint64_t packed = 0;
    pack_short_string(bytes, len, &packed);
    if (tag == LLKV_OP_STARTS_WITH && !ci) {
      // as a range of packed keys: the pattern's bytes on top, then anything — a key below `lo` with the same top bytes would
      // be a shorter string, one above `hi` differs in the top bytes
      const uint64_t rest = len == 0 ? ~0ull : ((1ull << (64 - 8 * len)) - 1);
      std::vector<Lit> run(2);
      run[0].lo = packed; run[0].hi = 0;
      run[1].lo = (packed & ~rest) | rest; run[1].hi = 0;
      emit(OP_PRED_U, (uint8_t)(LLKV_BOUND_INCLUDED | (LLKV_BOUND_INCLUDED << 2)), 0, add_lit_run(run));
      return;
    }
    const uint8_t mode = tag == LLKV_OP_ENDS_WITH ? 0 : tag == LLKV_OP_CONTAINS ? 1 : 2;
    emit(OP_PRED_STR, (uint8_t)(mode | (ci ? 4 : 0)), (uint8_t)len, add_lit(packed, 0));
  }

  void emit_in_leaf(const ColumnMeta& c, const llkv_literal* l, int n) {
    const int dom = col_domain(c);
    std::vector<Lit> run;
    uint16_t opc = OP_IN_BITS;
    if (dom == DOM_DEC) {
      opc = OP_IN_D;
      int ds = c.scale;
      for (int i = 0; i < n; ++i)
        if (l[i].kind == LLKV_LIT_DECIMAL128 && l[i].scale > ds) ds = l[i].scale;
      const i128 f = pow10_i128(ds - c.scale);
      for (int i = 0; i < n; ++i) {
        const i128 r = dec_literal(l[i], ds);
        if (r % f != 0) continue;  // no value of the column's scale equals it
        need_wide_for(r / f);
        run.push_back(mk_lit_i(r / f));
      }
    } else {
      if (dom == DOM_F64 || dom == DOM_F32) opc = OP_IN_F;
      for (int i = 0; i < n; ++i) {
        Lit v = native_literal(c, dom, l[i]);
        v.hi = 0;  // OP_IN_BITS compares the low 64 bits
        run.push_back(v);
      }
    }
    if (run.size() > 255) fail(LLKV_ERR_INVALID_ARGUMENT, "IN list longer than 255 entries");
    const uint32_t first = run.empty() ? 0 : add_lit_run(run);
    emit(opc, 0, (uint8_t)run.size(), first);
  }

  // ---- arrow-mode scalar expressions ---------------------------------------------------------------------------
  void check_node(int idx) const {
    if (idx < 0 || idx >= n_nodes_) fail(LLKV_ERR_INTERNAL, "expression node %d out of range", idx);
  }
  const ColumnMeta& node_col(const llkv_scalar_node& nd, int* ci_out = nullptr) const {
    const int ci = find_col(nd.field_id);
    if (ci < 0) fail(LLKV_ERR_INTERNAL, "missing column for field %llu", (unsigned long long)nd.field_id);
    if (ci_out) *ci_out = ci;
    return req_.cols[ci];
  }

  DT infer_type(int idx) const {  // eval.rs:71-148
    check_node(idx);
    const llkv_scalar_node& nd = nodes_[idx];
    switch (nd.tag) {
      case LLKV_SE_COLUMN: {
        const ColumnMeta& c = node_col(nd);
        return dt(c.type, c.precision, c.scale);
      }
      case LLKV_SE_LITERAL: return literal_type(nd.literal);
      case LLKV_SE_BINARY: return common_type(infer_type(nd.left), infer_type(nd.right));
      case LLKV_SE_COMPARE: case LLKV_SE_NOT: case LLKV_SE_IS_NULL: return dt(LLKV_PT_BOOLEAN);
      case LLKV_SE_CAST: return dt(nd.cast_type, nd.cast_precision, nd.cast_scale);
      default: fail(LLKV_ERR_INTERNAL, "scalar node tag %d is not supported on this path", nd.tag);
    }
  }

  bool fast_numeric_ok(int idx, DT* out) const {  // fast_numeric.rs:40-60,250-300
    check_node(idx);
    const llkv_scalar_node& nd = nodes_[idx];
    switch (nd.tag) {
      case LLKV_SE_COLUMN: {
        const int ci = find_col(nd.field_id);
        if (ci < 0) return false;
        const ColumnMeta& c = req_.cols[ci];
        if (!(is_int_t(c.type) || is_float_t(c.type))) return false;
        *out = dt(c.type);
        return true;
      }
      case LLKV_SE_LITERAL:
        if (nd.literal.kind == LLKV_LIT_INT128 || nd.literal.kind == LLKV_LIT_NULL || nd.literal.kind == LLKV_LIT_DECIMAL128) {
          *out = dt(LLKV_PT_INT64);
          return true;
        }
        if (nd.literal.kind == LLKV_LIT_FLOAT64) { *out = dt(LLKV_PT_FLOAT64); return true; }
        return false;
      case LLKV_SE_BINARY: {
        if (nd.op == LLKV_BIN_DIV || nd.op > LLKV_BIN_MOD) return false;
        DT l, r;
        if (!fast_numeric_ok(nd.left, &l) || !fast_numeric_ok(nd.right, &r)) return false;
        *out = common_type(l, r);
        return is_int_t(out->type) || is_float_t(out->type);
      }
      default: return false;
    }
  }

  // emits the cast of the top-of-stack value; the caller checked cast_supported
  void emit_cast(DT from, DT to) {
    if (dt_eq(from, to)) return;
    const Kind ik = kind_of_type(from.type), ok = kind_of_type(to.type);
    if (ik == K_NULL) {
      emit(OP_POP, 0, 0, 0);
      popped();
      push_null();
      return;
    }
    if ((ik == K_I64 || ik == K_DATE32 || ik == K_U64) && ok == K_DEC) {
      emit(OP_CAST_I_D, (uint8_t)to.s, (uint8_t)to.p, ik == K_U64 ? 1u : 0u);
      set_top_nullable(true);
      can_narrow_fail_ = true;
    } else if (ik == K_DEC && ok == K_DEC) {
      if (to.s >= from.s) {
        emit(OP_CAST_D_UP, (uint8_t)(to.s - from.s), (uint8_t)to.p, 0);
        can_narrow_fail_ = true;
      } else {
        emit(OP_CAST_D_DOWN, (uint8_t)(from.s - to.s), (uint8_t)to.p, 0);
        if (from.s - to.s > 18) wide_ = true;
      }
      set_top_nullable(true);
    } else if (ik == K_DEC && ok == K_F64) {
      emit(OP_CAST_D_F, 0, 0, add_lit(f64_bits(powi_f64(10.0, from.s)), 0));
    } else if ((ik == K_I64 || ik == K_DATE32) && ok == K_F64) {
      emit(OP_CAST_I_F, 0, 0, 0);
    } else if (ik == K_U64 && ok == K_F64) {
      emit(OP_CAST_U_F, 0, 0, 0);
    } else if (ik == K_F64 && ok == K_I64) {
      emit(OP_CAST_F_I, 0, 0, 0);
      set_top_nullable(true);
    } else if ((ik == K_I64 || ik == K_DATE32) && ok == K_I64) {
      const int bits = type_bits(to.type);
      if (bits < 64) {
        emit(OP_CAST_I_I, (uint8_t)bits, 0, 0);
        set_top_nullable(true);
      }
    } else if (ik == K_U64 && ok == K_I64) {
      emit(OP_CAST_U_I, 0, 0, 0);
      set_top_nullable(true);
    } else if (ik == K_I64 && ok == K_U64) {
      emit(OP_CAST_I_U, 0, 0, 0);
      set_top_nullable(true);
    } else if (ik == K_BOOL && ok == K_I64) {
      // 0/1 already
    } else if (ik == K_I64 && ok == K_BOOL) {
      emit(OP_CAST_I_B, 0, 0, 0);
    } else if (ik == K_F64 && ok == K_F64) {
      // stored as f64 either way
    } else {
      fail(LLKV_ERR_INTERNAL, "cast %d -> %d is not supported on this path", from.type, to.type);
    }
  }
  void hard_cast(DT from, DT to) {
    if (!cast_supported(from, to)) fail(LLKV_ERR_INTERNAL, "cast %d -> %d is not supported on this path", from.type, to.type);
    emit_cast(from, to);
  }

  // arithmetic on two equal-typed stack entries (arrow-arith numeric::*), result type returned
  DT emit_arith(DT l, DT r, int op) {
    const Kind k = kind_of_type(l.type);
    if (k == K_NULL) {
      emit(OP_POP, 0, 0, 0);
      popped();
      emit(OP_POP, 0, 0, 0);
      popped();
      push_null();
      return dt(LLKV_PT_NULL);
    }
    const bool n = nullable_[nullable_.size() - 1] || nullable_[nullable_.size() - 2] || op == LLKV_BIN_DIV;
    if (k == K_DEC) {
      const DT rt = arith_type(l, r, op);
      binary(op == LLKV_BIN_ADD ? OP_ADD_D : op == LLKV_BIN_SUB ? OP_SUB_D : OP_MUL_D, 0, 0, n);
      can_narrow_fail_ = true;
      return rt;
    }
    if (k == K_I64) {
      static const uint16_t ops[5] = {OP_ADD_I, OP_SUB_I, OP_MUL_I, OP_DIV_I, OP_MOD_I};
      binary(ops[op], 0, 0, n);
      return l;
    }
    if (k == K_F64) {
      static const uint16_t ops[5] = {OP_ADD_F, OP_SUB_F, OP_MUL_F, OP_DIV_F, OP_MOD_F};
      binary(ops[op], 0, 0, n);
      return l;
    }
    fail(LLKV_ERR_INTERNAL, "arithmetic on type %d is not supported on this path", l.type);
  }

  // result type of try_evaluate_vectorized without emitting (needed to cast the lhs before the rhs is pushed)
  VecInfo vec_type(int idx) const {
    check_node(idx);
    const llkv_scalar_node& nd = nodes_[idx];
    VecInfo v;
    switch (nd.tag) {
      case LLKV_SE_COLUMN: {
        const ColumnMeta& c = node_col(nd);
        v.t = dt(c.type, c.precision, c.scale);
        return v;
      }
      case LLKV_SE_LITERAL:
        v.t = literal_type(nd.literal);
        v.scalar = true;
        return v;
      case LLKV_SE_BINARY: {
        if (nd.op > LLKV_BIN_MOD) fail(LLKV_ERR_INTERNAL, "binary op %d is not supported on this path", nd.op);
        const VecInfo l = vec_type(nd.left), r = vec_type(nd.right);
        const DT ct = common_type(l.t, r.t);
        if (!cast_supported(l.t, ct) || !cast_supported(r.t, ct))
          fail(LLKV_ERR_INTERNAL, "cast to common type %d is not supported on this path", ct.type);
        const Kind k = kind_of_type(ct.type);
        if (k == K_NULL) v.t = dt(LLKV_PT_NULL);
        else if (k == K_DEC) v.t = arith_type(ct, ct, nd.op);
        else if (k == K_I64 || k == K_F64) v.t = ct;
        else fail(LLKV_ERR_INTERNAL, "arithmetic on type %d is not supported on this path", ct.type);
        v.scalar = l.scalar && r.scalar;
        return v;
      }
      case LLKV_SE_CAST: {
        const VecInfo in = vec_type(nd.left);
        v.t = dt(nd.cast_type, nd.cast_precision, nd.cast_scale);
        if (!cast_supported(in.t, v.t)) fail(LLKV_ERR_INTERNAL, "cast %d -> %d is not supported on this path", in.t.type, v.t.type);
        v.scalar = in.scalar;
        return v;
      }
      case LLKV_SE_COMPARE: {
        const VecInfo l = vec_type(nd.left), r = vec_type(nd.right);
        v.t = dt(LLKV_PT_BOOLEAN);
        v.scalar = l.scalar && r.scalar;
        return v;
      }
      default: fail(LLKV_ERR_INTERNAL, "scalar node tag %d is not supported on this path", nd.tag);
    }
  }

  void push_literal_value(const llkv_literal& l) {  // literal_to_array (eval.rs:521-543)
    switch (l.kind) {
      case LLKV_LIT_BOOLEAN: push_lit_bits(l.lo != 0); break;
      case LLKV_LIT_INT128: push_lit_i((i128)(int64_t)lit_i128(l)); break;
      case LLKV_LIT_FLOAT64: push_lit_bits(l.lo); break;
      case LLKV_LIT_DECIMAL128: push_lit_i(lit_i128(l)); break;
      case LLKV_LIT_DATE32: push_lit_i((i128)(int64_t)l.lo); break;
      case LLKV_LIT_STRING: {
        const char* bytes;
        size_t len;
        literal_bytes(l, &bytes, &len);
        uint64_t k = 0;
        pack_short_string((const uint8_t*)bytes, (uint32_t)std::min<size_t>(len, 7), &k);
        push_lit_bits(k);
        break;
      }
      default: push_null(); break;
    }
  }

  VecInfo emit_vec(int idx) {  // try_evaluate_vectorized (eval.rs:616-750)
    const llkv_scalar_node& nd = nodes_[idx];
    const VecInfo me = vec_type(idx);
    switch (nd.tag) {
      case LLKV_SE_COLUMN: {
        int ci;
        node_col(nd, &ci);
        push_col(ci);
        break;
      }
      case LLKV_SE_LITERAL: push_literal_value(nd.literal); break;
      case LLKV_SE_BINARY: {
        const VecInfo l = vec_type(nd.left), r = vec_type(nd.right);
        const DT ct = common_type(l.t, r.t);
        emit_vec(nd.left);
        emit_cast(l.t, ct);
        emit_vec(nd.right);
        emit_cast(r.t, ct);
        emit_arith(ct, ct, nd.op);
        break;
      }
      case LLKV_SE_CAST: {
        const VecInfo in = emit_vec(nd.left);
        emit_cast(in.t, me.t);
        break;
      }
      case LLKV_SE_COMPARE: {
        emit_compare(nd.left, nd.op, nd.right, /*batch=*/false);
        break;
      }
      default: fail(LLKV_ERR_INTERNAL, "scalar node tag %d is not supported on this path", nd.tag);
    }
    return me;
  }

  // NumericFastPath::execute (fast_numeric.rs:250-356): every leaf is cast to the target type first
  void emit_fast(int idx, DT target) {
    const llkv_scalar_node& nd = nodes_[idx];
    const Kind tk = kind_of_type(target.type);
    switch (nd.tag) {
      case LLKV_SE_COLUMN: {
        int ci;
        const ColumnMeta& c = node_col(nd, &ci);
        push_col(ci);
        hard_cast(dt(c.type, c.precision, c.scale), target);
        break;
      }
      case LLKV_SE_LITERAL: {
        const llkv_literal& l = nd.literal;
        if (l.kind == LLKV_LIT_NULL) { push_null(); break; }
        if (tk == K_F64) push_lit_bits(f64_bits(l.kind == LLKV_LIT_FLOAT64 ? lit_f64(l) : (double)lit_i128(l)));
        else if (tk == K_I64) {
          if (l.kind == LLKV_LIT_FLOAT64) fail(LLKV_ERR_INTERNAL, "float literal in integer fast path");
          const i128 v = lit_i128(l);
          if (!fits_i64(v)) fail(LLKV_ERR_INVALID_ARGUMENT, "literal out of range for Int64");
          push_lit_i(v);
        } else fail(LLKV_ERR_INTERNAL, "fast path target %d is not supported on this path", target.type);
        break;
      }
      default:
        emit_fast(nd.left, target);
        emit_fast(nd.right, target);
        emit_arith(target, target, nd.op);
        break;
    }
  }

  // ScalarEvaluator::evaluate_batch_simplified (eval.rs:565-614)
  DT emit_batch_arrow(int root) {
    const DT pref = infer_type(root);
    DT fo;
    if ((is_int_t(pref.type) || is_float_t(pref.type)) && fast_numeric_ok(root, &fo) && dt_eq(fo, pref)) {
      emit_fast(root, pref);
      return pref;
    }
    const VecInfo v = emit_vec(root);
    if (v.scalar) return v.t;
    if (dt_eq(v.t, pref)) return v.t;
    if (cast_supported(v.t, pref)) {  // cast(..).unwrap_or(array)
      emit_cast(v.t, pref);
      return pref;
    }
    return v.t;
  }

  // string comparisons inside scalar expressions work on packed short strings; dictionary codes of different columns (or a
  // code and a packed literal) do not compare
  void reject_dict_columns() const {
    for (const ColumnMeta& c : req_.cols)
      if (c.dict_sorted && c.type == LLKV_PT_UTF8)
        for (int i = 0; i < n_nodes_; ++i)
          if (nodes_[i].tag == LLKV_SE_COLUMN && find_col(nodes_[i].field_id) >= 0 && &req_.cols[find_col(nodes_[i].field_id)] == &c)
            fail(LLKV_ERR_INVALID_ARGUMENT, "scalar expressions over a dictionary-coded (long string) column are not on this path: use a typed predicate");
  }

  // compute_compare (kernels.rs:269-297) over two sub-expressions -> B on the stack
  void emit_compare(int left, int cmp, int right, bool batch) {
    check_node(left);
    check_node(right);
    // the type each side will have is needed before the rhs is emitted
    DT lt, rt;
    rt = batch ? batch_type(right) : vec_type(right).t;
    lt = batch ? emit_batch_arrow(left) : emit_vec(left).t;
    const DT ct = common_type(lt, rt);
    hard_cast(lt, ct);
    const DT rt2 = batch ? emit_batch_arrow(right) : emit_vec(right).t;
    if (!dt_eq(rt, rt2)) fail(LLKV_ERR_INTERNAL, "compare: inconsistent rhs type inference");
    hard_cast(rt, ct);
    uint16_t opc;
    switch (kind_of_type(ct.type)) {
      case K_I64: case K_DATE32: opc = OP_CMP_I; break;
      case K_STR: reject_dict_columns(); opc = OP_CMP_U; break;
      case K_U64: case K_BOOL: opc = OP_CMP_U; break;
      case K_F64: opc = OP_CMP_F; break;
      case K_DEC: opc = OP_CMP_D; break;
      default: fail(LLKV_ERR_INTERNAL, "compare on type %d is not supported on this path", ct.type);
    }
    if (cmp < LLKV_CMP_EQ || cmp > LLKV_CMP_GE) fail(LLKV_ERR_INTERNAL, "bad compare op %d", cmp);
    const bool n = nullable_[nullable_.size() - 1] || nullable_[nullable_.size() - 2];
    binary(opc, (uint8_t)cmp, 0, n);
  }
  // result type of emit_batch_arrow without emitting
  DT batch_type(int root) const {
    const DT pref = infer_type(root);
    DT fo;
    if ((is_int_t(pref.type) || is_float_t(pref.type)) && fast_numeric_ok(root, &fo) && dt_eq(fo, pref)) return pref;
    const VecInfo v = vec_type(root);
    if (v.scalar) return v.t;
    if (dt_eq(v.t, pref)) return v.t;
    if (cast_supported(v.t, pref)) return pref;
    return v.t;
  }

  void emit_compare_leaf(int left, int cmp, int right) { emit_compare(left, cmp, right, /*batch=*/true); }

  // evaluate_in_list_over_rows (llkv-scan/src/predicate.rs:442-560)
  void emit_in_list_leaf(const llkv_eval_op& op) {
    const ProgramView& pg = *req_.prog;
    check_node(op.expr_left);
    if (op.child_count < 0 || op.expr_right < 0 || op.expr_right + op.child_count > pg.n_list_roots)
      fail(LLKV_ERR_INTERNAL, "IN list roots out of range");
    const DT tt = emit_batch_arrow(op.expr_left);
    emit(OP_BOOL_LIT, 0, 0, 0);  // accumulator: matched = 0, saw_null = 0
    pushed(false);
    for (int li = 0; li < op.child_count; ++li) {
      const int item = pg.list_roots[op.expr_right + li];
      check_node(item);
      const DT it = batch_type(item);
      const DT ct = common_type(tt, it);
      emit(OP_PICK, 1, 0, 0);  // copy of the target
      pushed(nullable_[nullable_.size() - 2]);
      hard_cast(tt, ct);
      const DT it2 = emit_batch_arrow(item);
      if (!dt_eq(it, it2)) fail(LLKV_ERR_INTERNAL, "IN list: inconsistent item type inference");
      hard_cast(it, ct);
      uint16_t opc;
      switch (kind_of_type(ct.type)) {
        case K_I64: case K_DATE32: opc = OP_CMP_I; break;
        case K_STR: reject_dict_columns(); opc = OP_CMP_U; break;
      case K_U64: case K_BOOL: opc = OP_CMP_U; break;
        case K_F64: opc = OP_CMP_F; break;
        case K_DEC: opc = OP_CMP_D; break;
        default: fail(LLKV_ERR_INTERNAL, "compare on type %d is not supported on this path", ct.type);
      }
      binary(opc, LLKV_CMP_EQ, 0, true);
      binary(OP_INLIST_FOLD, 0, 0, true);
    }
    binary(OP_INLIST_END, (uint8_t)(op.negated != 0), 0, true);
  }

  // ---- exact-mode scalar expressions (GROUP BY aggregates): PlanValue interpreter, llkv-executor/src/lib.rs:7008-7440
  struct ExactKind {
    int kind = 0;  // 0 Null, 1 Integer, 2 Float, 3 Decimal
    int scale = 0;
  };
  int reuse_node_ = -1;  // exact mode: this node's value is already on top of the stack (kept by the previous aggregate)
  ExactKind emit_exact(int idx) {
    check_node(idx);
    if (idx == reuse_node_) {
      reuse_node_ = -1;
      return exact_kind(idx);
    }
    const llkv_scalar_node& nd = nodes_[idx];
    ExactKind out;
    switch (nd.tag) {
      case LLKV_SE_COLUMN: {
        int ci;
        const ColumnMeta& c = node_col(nd, &ci);
        if (c.type == LLKV_PT_DECIMAL128) { out.kind = 3; out.scale = c.scale; }
        else if (is_float_t(c.type)) out.kind = 2;
        else if (type_is_unsigned_int(c.type) || type_is_signed_int(c.type)) out.kind = 1;
        else fail(LLKV_ERR_INVALID_ARGUMENT, "column type %d is not numeric in an aggregate expression", c.type);
        push_col(ci);
        return out;
      }
      case LLKV_SE_LITERAL: {
        const llkv_literal& l = nd.literal;
        if (l.kind == LLKV_LIT_INT128) { out.kind = 1; push_lit_i((i128)(int64_t)lit_i128(l)); }
        else if (l.kind == LLKV_LIT_FLOAT64) { out.kind = 2; push_lit_bits(l.lo); }
        else if (l.kind == LLKV_LIT_DECIMAL128) { out.kind = 3; out.scale = l.scale; push_lit_i(lit_i128(l)); }
        else if (l.kind == LLKV_LIT_NULL) { out.kind = 0; push_null(); }
        else fail(LLKV_ERR_INVALID_ARGUMENT, "literal kind %d is not supported in an exact aggregate expression", l.kind);
        return out;
      }
      case LLKV_SE_BINARY: {
        // types first (the lhs must be rescaled before the rhs is pushed)
        const ExactKind lk = exact_kind(nd.left), rk = exact_kind(nd.right);
        if (lk.kind == 0 || rk.kind == 0) {  // NULL propagates
          emit_exact(nd.left);
          emit_exact(nd.right);
          emit(OP_POP, 0, 0, 0);
          popped();
          emit(OP_POP, 0, 0, 0);
          popped();
          push_null();
          return out;
        }
        if (lk.kind == 3 || rk.kind == 3) {
          if (lk.kind == 2 || rk.kind == 2) fail(LLKV_ERR_INVALID_ARGUMENT, "Cannot perform exact decimal arithmetic with Float operands");
          if (nd.op > LLKV_BIN_MUL) fail(LLKV_ERR_INVALID_ARGUMENT, "decimal op %d is not supported in an exact aggregate expression", nd.op);
          const int sa = lk.kind == 3 ? lk.scale : 0, sb = rk.kind == 3 ? rk.scale : 0;
          can_narrow_fail_ = true;
          if (nd.op == LLKV_BIN_MUL) {
            const int t = sa + sb;
            if (t > 38 || t < -38) fail(LLKV_ERR_INVALID_ARGUMENT, "Decimal multiplication overflow");
            emit_exact(nd.left);
            emit_exact(nd.right);
            const bool n = nullable_[nullable_.size() - 1] || nullable_[nullable_.size() - 2];
            binary(OP_MUL_D, 0, 1, n);
            out.kind = 3;
            out.scale = t;
            return out;
          }
          const int t = sa > sb ? sa : sb;
          emit_exact(nd.left);
          if (t > sa) emit(OP_RESCALE_DX, (uint8_t)(t - sa), 0, 0);
          emit_exact(nd.right);
          if (t > sb) emit(OP_RESCALE_DX, (uint8_t)(t - sb), 0, 0);
          const bool n = nullable_[nullable_.size() - 1] || nullable_[nullable_.size() - 2];
          binary(nd.op == LLKV_BIN_ADD ? OP_ADD_D : OP_SUB_D, 0, 1, n);
          out.kind = 3;
          out.scale = t;
          return out;
        }
        if (lk.kind == 1 && rk.kind == 1) {
          if (nd.op > LLKV_BIN_MUL) fail(LLKV_ERR_INVALID_ARGUMENT, "integer op %d is not supported in an exact aggregate expression", nd.op);
          emit_exact(nd.left);
          emit_exact(nd.right);
          const bool n = nullable_[nullable_.size() - 1] || nullable_[nullable_.size() - 2];
          binary(nd.op == LLKV_BIN_ADD ? OP_ADD_I : nd.op == LLKV_BIN_SUB ? OP_SUB_I : OP_MUL_I, 0, 1, n);
          out.kind = 1;
          return out;
        }
        if (nd.op > LLKV_BIN_MUL) fail(LLKV_ERR_INVALID_ARGUMENT, "float op %d is not supported in an exact aggregate expression", nd.op);
        emit_exact(nd.left);
        if (lk.kind == 1) emit(OP_CAST_I_F, 0, 0, 0);
        emit_exact(nd.right);
        if (rk.kind == 1) emit(OP_CAST_I_F, 0, 0, 0);
        const bool n = nullable_[nullable_.size() - 1] || nullable_[nullable_.size() - 2];
        binary(nd.op == LLKV_BIN_ADD ? OP_ADD_F : nd.op == LLKV_BIN_SUB ? OP_SUB_F : OP_MUL_F, 0, 0, n);
        out.kind = 2;
        return out;
      }
      default: fail(LLKV_ERR_INTERNAL, "scalar node tag %d is not supported in an exact aggregate expression", nd.tag);
    }
  }
  ExactKind exact_kind(int idx) const {
    check_node(idx);
    const llkv_scalar_node& nd = nodes_[idx];
    ExactKind out;
    switch (nd.tag) {
      case LLKV_SE_COLUMN: {
        const ColumnMeta& c = node_col(nd);
        if (c.type == LLKV_PT_DECIMAL128) { out.kind = 3; out.scale = c.scale; }
        else if (is_float_t(c.type)) out.kind = 2;
        else out.kind = 1;
        return out;
      }
      case LLKV_SE_LITERAL:
        if (nd.literal.kind == LLKV_LIT_INT128) out.kind = 1;
        else if (nd.literal.kind == LLKV_LIT_FLOAT64) out.kind = 2;
        else if (nd.literal.kind == LLKV_LIT_DECIMAL128) { out.kind = 3; out.scale = nd.literal.scale; }
        return out;
      case LLKV_SE_BINARY: {
        const ExactKind l = exact_kind(nd.left), r = exact_kind(nd.right);
        if (l.kind == 0 || r.kind == 0) return out;
        if (l.kind == 3 || r.kind == 3) {
          const int sa = l.kind == 3 ? l.scale : 0, sb = r.kind == 3 ? r.scale : 0;
          out.kind = 3;
          out.scale = nd.op == LLKV_BIN_MUL ? sa + sb : (sa > sb ? sa : sb);
          return out;
        }
        out.kind = (l.kind == 1 && r.kind == 1) ? 1 : 2;
        return out;
      }
      default: fail(LLKV_ERR_INTERNAL, "scalar node tag %d is not supported in an exact aggregate expression", nd.tag);
    }
  }

  // ---- GROUP BY keys ------------------------------------------------------------------------------------------
  void emit_keys() {
    Plan& p = out_.plan;
    const int nk = (int)req_.key_fields.size();
    p.n_keys = (uint32_t)nk;
    if (nk == 0) return;
    if (nk > kMaxKeys) fail(LLKV_ERR_INVALID_ARGUMENT, "too many GROUP BY keys (max %d)", kMaxKeys);
    int total = 0;
    for (int k = 0; k < nk; ++k) {
      const int ci = find_col(req_.key_fields[k]);
      if (ci < 0) fail(LLKV_ERR_NOT_FOUND, "unknown GROUP BY field %llu", (unsigned long long)req_.key_fields[k]);
      const ColumnMeta& c = req_.cols[ci];
      KeyLayout kl;
      kl.field_id = c.field_id;
      kl.type = c.type;
      kl.nullable = c.nullable;
      if (type_is_signed_int(c.type) || type_is_unsigned_int(c.type) || c.type == LLKV_PT_BOOLEAN) {
        kl.kind = KK_INT;
        kl.is_signed = type_is_signed_int(c.type);
        int width = c.type == LLKV_PT_BOOLEAN ? 8 : type_bits(c.type);
        if (c.has_minmax) {
          const uint64_t range = c.max_bits - c.min_bits;  // same for both signednesses (mod 2^64)
          int b = 1;
          while (b < 64 && (range >> b)) ++b;
          kl.bits = (uint8_t)b;
          kl.min = c.min_bits;
        } else {
          kl.bits = (uint8_t)width;
          kl.min = 0;
        }
      } else if (c.type == LLKV_PT_UTF8 && c.dict_sorted) {  // dictionary codes: ranks 0 .. entries-1
        kl.kind = KK_INT;
        kl.dict = true;
        const uint64_t range = c.dict_sorted->empty() ? 0 : c.dict_sorted->size() - 1;
        int b = 1;
        while (b < 64 && (range >> b)) ++b;
        kl.bits = (uint8_t)b;
        kl.min = 0;
      } else if (c.type == LLKV_PT_UTF8) {
        kl.kind = KK_STR;
        kl.strlen = c.max_strlen;
        kl.bits = (uint8_t)(8 * c.max_strlen + 3);
      } else {
        fail(LLKV_ERR_INVALID_ARGUMENT, "GROUP BY does not support column type %d", c.type);
      }
      total += kl.bits + (kl.nullable ? 1 : 0);
      out_.keys.push_back(kl);
      push_col(ci);
    }
    if (nk == 1 && out_.keys[0].kind == KK_INT && total > 63) {
      p.single_wide_key = 1;
      out_.keys[0].bits = 64;
      out_.keys[0].min = 0;
    } else if (total > 64) {
      // wider than one word: group by a 64-bit hash of the keys' images; the runtime verifies it and reads the key values
      // back from the columns (plan.h: single_wide_key == 2)
      p.single_wide_key = 2;
      for (KeyLayout& kl : out_.keys) {
        kl.kind = KK_INT;
        kl.bits = 64;
        kl.min = 0;
      }
    }
    for (int k = 0; k < nk; ++k) {
      p.key_bits[k] = out_.keys[k].bits;
      p.key_nullable[k] = out_.keys[k].nullable;
      p.key_kind[k] = out_.keys[k].kind;
      p.key_strlen[k] = out_.keys[k].strlen;
      p.key_min[k] = out_.keys[k].min;
    }
    emit(OP_GROUP, (uint8_t)nk, 0, 0);
    for (int k = 0; k < nk; ++k) popped();
  }

  // ---- aggregates --------------------------------------------------------------------------------------------
  int new_gword(uint8_t cls) {
    if (gclass_.size() >= (size_t)kMaxWords) fail(LLKV_ERR_INVALID_ARGUMENT, "too many aggregate state words (max %d)", kMaxWords);
    gclass_.push_back(cls);
    return (int)gclass_.size() - 1;
  }
  int new_fast(uint8_t kind, int gword) {
    FastWord f;
    memset(&f, 0, sizeof(f));
    f.kind = kind;
    f.gword = (uint32_t)gword;
    fast_.push_back(f);
    return (int)fast_.size() - 1;
  }
  struct WordRef {
    int g = -1, f = -1;
  };
  // allocates `n` consecutive global words of a class (+ matching fast words)
  WordRef alloc_words(uint8_t fast_kind, uint8_t cls, int n, bool align2 = false) {
    if (align2 && (gclass_.size() & 1)) new_gword(WC_SUM);  // padding keeps 128-bit pairs 16-byte aligned
    WordRef w;
    w.g = new_gword(cls);
    for (int i = 1; i < n; ++i) new_gword(cls);
    w.f = new_fast(fast_kind, w.g);
    return w;
  }

  std::string signature(int idx) const {
    check_node(idx);
    const llkv_scalar_node& nd = nodes_[idx];
    char buf[160];
    switch (nd.tag) {
      case LLKV_SE_COLUMN: snprintf(buf, sizeof(buf), "c%llu", (unsigned long long)nd.field_id); return buf;
      case LLKV_SE_LITERAL:
        snprintf(buf, sizeof(buf), "l%d:%d:%llx:%llx", nd.literal.kind, nd.literal.scale, (unsigned long long)nd.literal.lo,
                 (unsigned long long)nd.literal.hi);
        return buf;
      case LLKV_SE_BINARY: case LLKV_SE_COMPARE:
        snprintf(buf, sizeof(buf), "%c%d(", nd.tag == LLKV_SE_BINARY ? 'b' : 'q', nd.op);
        return std::string(buf) + signature(nd.left) + "," + signature(nd.right) + ")";
      case LLKV_SE_CAST:
        snprintf(buf, sizeof(buf), "k%d:%d:%d(", nd.cast_type, nd.cast_precision, nd.cast_scale);
        return std::string(buf) + signature(nd.left) + ")";
      default: snprintf(buf, sizeof(buf), "t%d#%d", nd.tag, idx); return buf;
    }
  }

  static int acc_kind_for(const llkv_agg_spec& sp) {  // new_with_projection_index (llkv-aggregate/src/lib.rs:463-748)
    if (sp.distinct) fail(LLKV_ERR_INVALID_ARGUMENT, "DISTINCT aggregates are outside this path");
    const int t = sp.data_type;
    switch (sp.kind) {
      case LLKV_AGG_COUNT: return sp.expr_root < 0 ? ACC_COUNT_STAR : ACC_COUNT_COL;
      case LLKV_AGG_COUNT_NULLS: return ACC_COUNT_NULLS;
      case LLKV_AGG_SUM: case LLKV_AGG_TOTAL: case LLKV_AGG_AVG: {
        const int base = sp.kind == LLKV_AGG_SUM ? ACC_SUM_I64 : sp.kind == LLKV_AGG_TOTAL ? ACC_TOTAL_I64 : ACC_AVG_I64;
        if (t == LLKV_PT_INT64) return base;
        if (t == LLKV_PT_DECIMAL128) return base + 2;
        if (t == LLKV_PT_FLOAT64 || t == LLKV_PT_UTF8) return base + 1;
        fail(LLKV_ERR_INVALID_ARGUMENT, "%s aggregate not supported for column type %d",
             sp.kind == LLKV_AGG_SUM ? "SUM" : sp.kind == LLKV_AGG_TOTAL ? "TOTAL" : "AVG", t);
      }
      case LLKV_AGG_MIN: case LLKV_AGG_MAX: {
        const int base = sp.kind == LLKV_AGG_MIN ? ACC_MIN_I64 : ACC_MAX_I64;
        if (t == LLKV_PT_INT64) return base;
        if (t == LLKV_PT_DECIMAL128) return base + 2;
        if (t == LLKV_PT_FLOAT64 || t == LLKV_PT_UTF8) return base + 1;
        fail(LLKV_ERR_INVALID_ARGUMENT, "%s aggregate not supported for column type %d", sp.kind == LLKV_AGG_MIN ? "MIN" : "MAX", t);
      }
    }
    fail(LLKV_ERR_INVALID_ARGUMENT, "unknown aggregate kind %d", sp.kind);
  }

  // type of the argument array the accumulator is fed (eval_agg_arg), without emitting
  DT arg_type(const llkv_agg_spec& sp) const {
    if (sp.expr_root < 0) return dt(LLKV_PT_NULL);
    check_node(sp.expr_root);
    const llkv_scalar_node& nd = nodes_[sp.expr_root];
    if (nd.tag == LLKV_SE_COLUMN) {
      const ColumnMeta& c = node_col(nd);
      return dt(c.type, c.precision, c.scale);
    }
    if (req_.expr_mode == LLKV_EXPR_EXACT) {
      const ExactKind k = exact_kind(sp.expr_root);
      return k.kind == 3 ? dt(LLKV_PT_DECIMAL128, 38, k.scale) : k.kind == 2 ? dt(LLKV_PT_FLOAT64) : k.kind == 1 ? dt(LLKV_PT_INT64) : dt(LLKV_PT_NULL);
    }
    return batch_type(sp.expr_root);
  }
  void emit_arg(const llkv_agg_spec& sp) {
    const llkv_scalar_node& nd = nodes_[sp.expr_root];
    if (nd.tag == LLKV_SE_COLUMN) {
      int ci;
      node_col(nd, &ci);
      push_col(ci);
    } else if (req_.expr_mode == LLKV_EXPR_EXACT) {
      emit_exact(sp.expr_root);
    } else {
      emit_batch_arrow(sp.expr_root);
    }
  }

  void emit_aggregates() {
    Plan& p = out_.plan;
    nodes_ = req_.agg_nodes;
    n_nodes_ = req_.n_agg_nodes;
    const bool grouped = p.n_keys != 0;
    // word 0: rows folded into the group (COUNT(*), occupancy of the special rows when partial tables are merged)
    const WordRef rows = alloc_words(FK_COUNT, WC_SUM, 1);
    emit(OP_AGG_COUNT_STAR, 0, (uint8_t)rows.f, (uint32_t)rows.g);
    if (grouped) {
      const WordRef first = alloc_words(FK_MIN, WC_MIN, 1);
      emit(OP_AGG_FIRSTROW, 0, (uint8_t)first.f, (uint32_t)first.g);
    }
    out_.aggs.resize((size_t)req_.n_aggs);
    for (int a = 0; a < req_.n_aggs; ++a) {
      const llkv_agg_spec& sp = req_.specs[a];
      AggLayout& L = out_.aggs[(size_t)a];
      L.acc = acc_kind_for(sp);
      L.precision = sp.precision;
      L.scale = sp.scale;
      if (L.acc == ACC_COUNT_STAR) {
        L.w_count = rows.g;
        continue;
      }
      // errors below are what the reference raises from update(): only if a row reaches the accumulator
      const size_t code_mark = code_.size(), lits_mark = lits_.size(), g_mark = gclass_.size(), f_mark = fast_.size();
      const std::vector<bool> stack_mark = nullable_;
      const std::map<std::string, int> facts_mark = facts_;
      const bool wide_mark = wide_, cnf_mark = can_narrow_fail_;
      // common prefix: when the next aggregate's argument is `this argument <op> something`, the value stays on the stack
      // (TPC-H Q1: sum(price*(1-disc)) then sum(price*(1-disc)*(1+tax)))
      bool keep_for_next = false;
      int next_left = -1;
      if (req_.expr_mode == LLKV_EXPR_EXACT && a + 1 < req_.n_aggs && sp.expr_root >= 0 && req_.specs[a + 1].expr_root >= 0 &&
          nodes_[sp.expr_root].tag == LLKV_SE_BINARY && nodes_[req_.specs[a + 1].expr_root].tag == LLKV_SE_BINARY) {
        next_left = nodes_[req_.specs[a + 1].expr_root].left;
        if (next_left >= 0 && next_left < n_nodes_ && signature(next_left) == signature(sp.expr_root) && reuse_node_ < 0) keep_for_next = true;
      }
      const bool had_reuse = reuse_node_ >= 0;
      try {
        emit_one_aggregate(sp, L, rows.g, keep_for_next);
        if (had_reuse && reuse_node_ >= 0) {  // the kept value was not needed after all
          reuse_node_ = -1;
          emit(OP_POP, 0, 0, 0);
          popped();
        }
        if (keep_for_next) {
          if (kept_on_stack_) reuse_node_ = next_left;
          kept_on_stack_ = false;
        }
      } catch (const CompileError& e) {
        reuse_node_ = -1;
        kept_on_stack_ = false;
        code_.resize(code_mark);
        lits_.resize(lits_mark);
        gclass_.resize(g_mark);
        fast_.resize(f_mark);
        nullable_ = stack_mark;
        facts_ = facts_mark;
        wide_ = wide_mark;
        can_narrow_fail_ = cnf_mark;
        L.raise_code = e.code;
        L.raise_message = e.msg;
        L.dead = true;
        emit(OP_RAISE, 6 /* FLAG_TYPE_ERROR bit */, 0, 0);
      }
    }
  }

  struct Fact {
    const char* name;
    uint16_t op;
    uint8_t fast_kind, cls;
    int n_words;
    bool align2;
    bool after_numeric_cast;  // operates on the array_value_to_numeric (f64) image of the argument
  };

  bool kept_on_stack_ = false;
  void emit_one_aggregate(const llkv_agg_spec& sp, AggLayout& L, int rows_word, bool keep_for_next = false) {
    check_node(sp.expr_root);
    const DT at = arg_type(sp);
    const Kind ak = kind_of_type(at.type);
    const std::string sig = (req_.expr_mode == LLKV_EXPR_EXACT ? "x:" : "a:") + signature(sp.expr_root);
    const int acc = L.acc;

    // which accumulator family, and whether it accepts this array type (acc_update in the reference)
    const bool fam_i = acc == ACC_SUM_I64 || acc == ACC_TOTAL_I64 || acc == ACC_AVG_I64 || acc == ACC_MIN_I64 || acc == ACC_MAX_I64;
    const bool fam_f = acc == ACC_SUM_F64 || acc == ACC_TOTAL_F64 || acc == ACC_AVG_F64 || acc == ACC_MIN_F64 || acc == ACC_MAX_F64;
    const bool fam_d = acc == ACC_SUM_DEC || acc == ACC_TOTAL_DEC || acc == ACC_AVG_DEC || acc == ACC_MIN_DEC || acc == ACC_MAX_DEC;
    bool dead = false;
    if (fam_i) {
      if (ak == K_NULL) dead = true;
      else if (at.type != LLKV_PT_INT64) fail(LLKV_ERR_INVALID_ARGUMENT, "aggregate expected an INT column in execution");
    } else if (fam_f) {
      if (ak == K_NULL) dead = true;
      else if (!((ak == K_I64 && at.type == LLKV_PT_INT64) || (ak == K_F64 && at.type == LLKV_PT_FLOAT64) || ak == K_DEC || ak == K_BOOL))
        fail(LLKV_ERR_INVALID_ARGUMENT, "Numeric coercion not supported for column type %d", at.type);
    } else if (fam_d) {
      if (ak != K_DEC) fail(LLKV_ERR_INVALID_ARGUMENT, "Expected Decimal128 array");
    } else if (ak == K_NULL) {
      dead = true;  // COUNT(col) / CountNulls over a NULL-typed array: no valid values
    }
    L.dead = dead;
    L.all_null_group_is_error = fam_d && req_.expr_mode == LLKV_EXPR_EXACT && req_.key_fields.size() > 0 &&
                                nodes_[sp.expr_root].tag != LLKV_SE_COLUMN;

    // facts this accumulator needs
    std::vector<Fact> need;
    const Fact f_count = {"count", OP_AGG_COUNT, FK_COUNT, WC_SUM, 1, false, false};
    const Fact f_sum_i = {"sum_i", OP_AGG_SUM_I, FK_SUM_I64, WC_SUM, 2, false, false};
    const Fact f_sum_d = {"sum_d", OP_AGG_SUM_D, FK_SUM_I128, WC_SUM, 4, false, false};
    const Fact f_min_i = {"min_i", OP_AGG_MIN_I, FK_MIN, WC_MIN, 1, false, false};
    const Fact f_max_i = {"max_i", OP_AGG_MAX_I, FK_MAX, WC_MAX, 1, false, false};
    const Fact f_min_d = {"min_d", OP_AGG_MIN_D, FK_MIN128_HI, WC_MIN128, 2, true, false};
    const Fact f_max_d = {"max_d", OP_AGG_MAX_D, FK_MAX128_HI, WC_MAX128, 2, true, false};
    const Fact f_fsum = {"fsum", OP_AGG_FSUM, FK_FSUM, WC_FSUM, 1, false, true};
    const Fact f_min_f = {"min_f", OP_AGG_MIN_F, FK_MIN, WC_MIN, 1, false, true};
    const Fact f_max_f = {"max_f", OP_AGG_MAX_F, FK_MAX, WC_MAX, 1, false, true};
    const Fact f_fvalid = {"first_valid", OP_AGG_FIRSTVALID, FK_MIN, WC_MIN, 1, false, true};
    const Fact f_fnan = {"first_nan", OP_AGG_FIRSTNAN, FK_MIN, WC_MIN, 1, false, true};
    if (!dead) {
      switch (acc) {
        case ACC_COUNT_COL: case ACC_COUNT_NULLS: need = {f_count}; break;
        case ACC_SUM_I64: case ACC_AVG_I64: need = {f_count, f_sum_i}; break;
        case ACC_TOTAL_I64: need = {f_count, f_fsum}; break;
        case ACC_MIN_I64: need = {f_count, f_min_i}; break;
        case ACC_MAX_I64: need = {f_count, f_max_i}; break;
        case ACC_SUM_F64: case ACC_TOTAL_F64: case ACC_AVG_F64: need = {f_count, f_fsum}; break;
        case ACC_MIN_F64: need = {f_fvalid, f_fnan, f_min_f}; break;
        case ACC_MAX_F64: need = {f_fvalid, f_fnan, f_max_f}; break;
        case ACC_SUM_DEC: case ACC_TOTAL_DEC: case ACC_AVG_DEC: need = {f_count, f_sum_d}; break;
        case ACC_MIN_DEC: need = {f_count, f_min_d}; break;
        case ACC_MAX_DEC: need = {f_count, f_max_d}; break;
      }
    }
    if (dead) {
      // the argument is still evaluated by the reference (errors inside it would surface): keep that, drop the value
      if (sp.expr_root >= 0 && nodes_[sp.expr_root].tag != LLKV_SE_COLUMN) {
        emit_arg(sp);
        emit(OP_POP, 0, 0, 0);
        popped();
      }
      return;
    }

    // a count over an argument that can never be NULL is the group's row count
    // (decided after emission: static nullability comes out of emit_arg)
    std::vector<Fact> missing;
    for (const Fact& f : need)
      if (!facts_.count(sig + "|" + f.name)) missing.push_back(f);

    if (!missing.empty()) {
      emit_arg(sp);
      const bool arg_nullable = get_top_nullable();
      // raw-domain facts first, then the numeric (f64) image
      bool casted = false;
      std::vector<Fact> ordered;
      for (const Fact& f : missing) if (!f.after_numeric_cast) ordered.push_back(f);
      for (const Fact& f : missing) if (f.after_numeric_cast) ordered.push_back(f);
      // drop the count if it aliases the row count
      std::vector<Fact> todo;
      for (const Fact& f : ordered) {
        if (!strcmp(f.name, "count") && !arg_nullable) {
          facts_[sig + "|count"] = rows_word;
          continue;
        }
        todo.push_back(f);
      }
      for (size_t i = 0; i < todo.size(); ++i) {
        const Fact& f = todo[i];
        if (f.after_numeric_cast && !casted) {
          if (ak == K_I64) emit(OP_CAST_I_F, 0, 0, 0);
          else if (ak == K_DEC) emit(OP_CAST_D_F, 0, 0, add_lit(f64_bits(powi_f64(10.0, at.s)), 0));
          else if (ak == K_BOOL) emit(OP_CAST_U_F, 0, 0, 0);
          casted = true;
        }
        const WordRef w = alloc_words(f.fast_kind, f.cls, f.n_words, f.align2);
        if (f.n_words == 2 && f.align2) {  // 128-bit min/max: second word of the pair
          gclass_[(size_t)w.g + 1] = f.cls == WC_MIN128 ? WC_PAIR_LO_MIN : WC_PAIR_LO_MAX;
          new_fast(FK_SKIP, w.g + 1);
        }
        facts_[sig + "|" + f.name] = w.g;
        const bool keep = i + 1 < todo.size() || keep_for_next;
        emit(f.op, keep ? 1 : 0, (uint8_t)w.f, (uint32_t)w.g);
      }
      if (keep_for_next && !casted) {
        kept_on_stack_ = true;  // raw value stays for the next aggregate
      } else {
        if (todo.empty() || (keep_for_next && casted)) emit(OP_POP, 0, 0, 0);
        popped();
      }
    }
    auto fact = [&](const char* name) -> int {
      auto it = facts_.find(sig + "|" + name);
      return it == facts_.end() ? -1 : it->second;
    };
    L.w_count = fact("count");
    switch (acc) {
      case ACC_SUM_I64: case ACC_AVG_I64: L.w_val = fact("sum_i"); L.n_limbs = 2; break;
      case ACC_TOTAL_I64: case ACC_SUM_F64: case ACC_TOTAL_F64: case ACC_AVG_F64: L.w_val = fact("fsum"); break;
      case ACC_MIN_I64: L.w_val = fact("min_i"); break;
      case ACC_MAX_I64: L.w_val = fact("max_i"); break;
      case ACC_MIN_F64: L.w_val = fact("min_f"); L.w_first_valid = fact("first_valid"); L.w_first_nan = fact("first_nan"); break;
      case ACC_MAX_F64: L.w_val = fact("max_f"); L.w_first_valid = fact("first_valid"); L.w_first_nan = fact("first_nan"); break;
      case ACC_SUM_DEC: case ACC_TOTAL_DEC: case ACC_AVG_DEC: L.w_val = fact("sum_d"); L.n_limbs = 4; break;
      case ACC_MIN_DEC: L.w_val = fact("min_d"); break;
      case ACC_MAX_DEC: L.w_val = fact("max_d"); break;
      default: break;
    }
  }

  // ---- post passes ---------------------------------------------------------------------------------------------
  static bool can_raise(uint16_t op) {
    switch (op) {
      case OP_ADD_I: case OP_SUB_I: case OP_MUL_I: case OP_DIV_I: case OP_MOD_I:
      case OP_ADD_D: case OP_SUB_D: case OP_MUL_D: case OP_CAST_I_D: case OP_CAST_D_UP: case OP_RESCALE_DX:
        return true;
      default: return false;
    }
  }
  void mark_filter_exits() {
    // an OP_FILTER may stop the warp early only if nothing between it and the end of the selection phase can raise
    bool raises_later = false;
    for (size_t i = select_end_; i-- > 0;) {
      if (code_[i].op == OP_FILTER) code_[i].a = raises_later ? 0 : 1;
      if (can_raise(code_[i].op)) raises_later = true;
    }
  }

  void finish() {
    Plan& p = out_.plan;
    p.n_instr = (uint32_t)code_.size();
    for (size_t i = 0; i < code_.size(); ++i) p.code[i] = code_[i];
    p.n_lits = (uint32_t)lits_.size();
    for (size_t i = 0; i < lits_.size(); ++i) p.lits[i] = lits_[i];
    p.n_cols = (uint32_t)plan_cols_.size();
    uint32_t alg = 0, phys = 0;
    for (size_t i = 0; i < plan_cols_.size(); ++i) {
      const ColumnMeta& c = *plan_cols_[i];
      p.cols[i].base = c.dev_values;
      p.cols[i].validity = c.dev_validity;
      p.cols[i].elem_bytes = c.elem_bytes;
      alg += c.arrow_bytes;
      phys += c.elem_bytes;
    }
    p.max_depth = (uint32_t)max_sp_;
    p.txn_id = req_.mvcc.txn_id;
    p.snapshot_id = req_.mvcc.snapshot_id;
    p.n_noncommitted = (uint32_t)req_.mvcc.noncommitted.size();
    for (size_t i = 0; i < req_.mvcc.noncommitted.size() && i < (size_t)kMaxNoncommitted; ++i) p.noncommitted[i] = req_.mvcc.noncommitted[i];
    if (gclass_.size() & 1) new_gword(WC_SUM);  // even row stride keeps 128-bit pairs aligned in every row
    p.n_gwords = (uint32_t)gclass_.size();
    for (size_t i = 0; i < gclass_.size(); ++i) p.gword_class[i] = gclass_[i];
    p.n_fast_words = (uint32_t)fast_.size();
    for (size_t i = 0; i < fast_.size(); ++i) p.fast[i] = fast_[i];
    out_.wide = wide_;
    out_.can_narrow_fail = can_narrow_fail_ && !wide_;
    out_.algorithmic_bytes_per_row = alg;
    out_.physical_bytes_per_row = phys;
    out_.fast = false;
    p.n_finstr = 0;
    if (!req_.no_fast) {
      const size_t lits_mark = lits_.size();
      if (lower_fast()) {
        out_.fast = true;
        // the lean program raises FLAG_NARROW_FAIL only from its checked operations (everything else was proven to fit)
        bool checked = false;
        for (uint32_t i = 0; i < p.n_finstr; ++i) {
          const FInstr& fi = p.fcode[i];
          const uint32_t fb = fi.a & 0x7f;
          if ((fi.op == FO_OP_COL || fi.op == FO_OP_LIT || fi.op == FO_OP_TMP) && (fb == FB_ADD_CK || fb == FB_SUB_CK || fb == FB_MUL_CK)) checked = true;
        }
        out_.can_narrow_fail = checked;
        p.n_lits = (uint32_t)lits_.size();
        for (size_t i = 0; i < lits_.size(); ++i) p.lits[i] = lits_[i];
      } else {
        lits_.resize(lits_mark);
        p.n_finstr = 0;
      }
    }
  }

  // ---- lowering to the lean kernel (fast_kernel.cu) -----------------------------------------------------------------
  // Abstract interpretation of the generic program with value intervals from the columns' min/max statistics: when no
  // input can be NULL and every arithmetic result provably fits 64 bits (so no check can fire), the plan also gets a
  // FastOp program.  Anything outside the hot subset keeps only the generic program.
  struct Iv {
    bool known = false;  // integer interval [lo, hi] is valid
    i128 lo = 0, hi = 0;
    bool is_float = false;
  };
  static Iv iv_exact(i128 v) {
    Iv x;
    x.known = true;
    x.lo = x.hi = v;
    return x;
  }
  static bool iv_fits(const Iv& x, i128 lo, i128 hi) { return x.known && x.lo >= lo && x.hi <= hi; }
  static bool iv_fits_i64(const Iv& x) { return iv_fits(x, (i128)INT64_MIN, (i128)INT64_MAX); }
  static bool iv_fits_i32(const Iv& x) { return iv_fits(x, (i128)INT32_MIN, (i128)INT32_MAX); }
  static Iv iv_arith(int op, const Iv& a, const Iv& b) {  // 0 add, 1 sub, 2 mul
    Iv r;
    if (!a.known || !b.known) return r;
    i128 c[4];
    bool ov = false;
    if (op == 0) { ov |= __builtin_add_overflow(a.lo, b.lo, &c[0]); ov |= __builtin_add_overflow(a.hi, b.hi, &c[1]); c[2] = c[0]; c[3] = c[1]; }
    else if (op == 1) { ov |= __builtin_sub_overflow(a.lo, b.hi, &c[0]); ov |= __builtin_sub_overflow(a.hi, b.lo, &c[1]); c[2] = c[0]; c[3] = c[1]; }
    else {
      ov |= __builtin_mul_overflow(a.lo, b.lo, &c[0]);
      ov |= __builtin_mul_overflow(a.lo, b.hi, &c[1]);
      ov |= __builtin_mul_overflow(a.hi, b.lo, &c[2]);
      ov |= __builtin_mul_overflow(a.hi, b.hi, &c[3]);
    }
    if (ov) return r;
    r.known = true;
    r.lo = r.hi = c[0];
    for (int i = 1; i < 4; ++i) {
      if (c[i] < r.lo) r.lo = c[i];
      if (c[i] > r.hi) r.hi = c[i];
    }
    return r;
  }
  static i128 round_div(i128 x, i128 d) {  // half away from zero
    i128 q = x / d, rem = x % d, half = d / 2;
    if (x >= 0) { if (rem >= half) q += 1; } else { if (rem <= -half) q -= 1; }
    return q;
  }
  Iv column_interval(const ColumnMeta& c) const {
    Iv x;
    switch (c.load_kind) {
      case LK_F32: case LK_F64: x.is_float = true; return x;
      case LK_STR8: case LK_U64: case LK_D128: case LK_I64: break;
      default: break;
    }
    const bool is_signed = type_is_signed_int(c.type) || c.type == LLKV_PT_DECIMAL128;
    if (c.has_minmax) {
      x.known = true;
      x.lo = is_signed ? (i128)(int64_t)c.min_bits : (i128)c.min_bits;
      x.hi = is_signed ? (i128)(int64_t)c.max_bits : (i128)c.max_bits;
      return x;
    }
    if (c.type == LLKV_PT_UTF8) return x;
    const int bits = c.type == LLKV_PT_DECIMAL128 ? 64 : (c.type == LLKV_PT_BOOLEAN ? 8 : type_bits(c.type));
    x.known = true;
    if (is_signed) { x.lo = -((i128)1 << (bits - 1)); x.hi = ((i128)1 << (bits - 1)) - 1; }
    else { x.lo = 0; x.hi = ((i128)1 << bits) - 1; }
    return x;
  }

  // symbolic value-stack entry of the accumulator machine
  struct Sym {
    enum Where : uint8_t { ACC, COL, LIT, TMP } where = LIT;
    uint8_t col = 0, load = 0, tmp = 0;
    uint32_t lit = 0;
    Iv iv;
    uint32_t nm = 0;  // plan columns whose NULLs make this value NULL
  };

  // (LLKV_GPU_VERBOSE=2 names the line at which a plan left the lean lowering)
  static bool lf_fail(int line) {
    static const bool verbose = [] { const char* e = getenv("LLKV_GPU_VERBOSE"); return e && atoi(e) >= 2; }();
    if (verbose && line < 0) fprintf(stderr, "[llkv] lean lowering gave up at interpreter op %d\n", -line);
    else if (verbose) fprintf(stderr, "[llkv] lean lowering gave up at compiler.cpp:%d\n", line);
    return false;
  }
  bool lower_fast() {
    Plan& p = out_.plan;
    if (wide_ || req_.bitmap_mode) return lf_fail(__LINE__);
    if (plan_cols_.empty()) return lf_fail(__LINE__);  // nothing to stream (COUNT(*) without a filter): no tiles for the lean pipeline
    for (const ColumnMeta* c : plan_cols_) {
      if (c->load_kind == LK_D128 && !c->dec_fits_i64) return lf_fail(__LINE__);
    }
    std::vector<FInstr> f;
    std::vector<Sym> st;
    bool tmp_used[kFastTmps] = {false, false, false};
    int max_tmps = 0;
    bool ok = true;
    auto map_load = [&](uint8_t lk) -> uint32_t {  // physical layouts the lean kernel reads
      switch (lk) {
        case LK_I32: case LK_D32: return LKF_4;
        case LK_I64: case LK_U64: case LK_F64: case LK_D64: return LKF_8;
        case LK_D128: return LKF_16;
        case LK_U8: return LKF_1;
        case LK_STR8: return LKF_S1;
        case LK_I8: return LKF_1S;
        case LK_I16: return LKF_2;
        case LK_U16: return LKF_2U;
        case LK_U32: return LKF_4U;
        case LK_F32: return LKF_4F;
        default: ok = false; return LKF_8;
      }
    };
    auto femit = [&](uint16_t op, uint32_t a, uint32_t b, uint32_t c) {
      FInstr in;
      memset(&in, 0, sizeof(in));
      in.op = op;
      in.a = a;
      in.b = b;
      in.c = c;
      // a pending "acc = ..." load folds into the instruction that consumes it
      if (!f.empty() && (f.back().op == FO_LD_COL || f.back().op == FO_LD_LIT || f.back().op == FO_LD_TMP) && op != FO_LEAF &&
          op != FO_MVCC && op != FO_SELECT_DONE && op != FO_GROUP && op != FO_END && op != FO_LD_COL && op != FO_LD_LIT &&
          op != FO_LD_TMP && op != FO_COUNT_STAR && op != FO_FIRSTROW && (op < FO_VALID || op == FO_CMP)) {
        in.d = f.back().d;
        in.e = f.back().e;
        in.f = f.back().f;
        f.pop_back();
      }
      f.push_back(in);
    };
    auto femit_load = [&](uint16_t op, uint32_t d, uint32_t e, uint32_t ff) {
      FInstr in;
      memset(&in, 0, sizeof(in));
      in.op = op;
      in.d = d;
      in.e = e;
      in.f = ff;
      f.push_back(in);
    };
    auto free_sym = [&](const Sym& x) {
      if (x.where == Sym::TMP) tmp_used[x.tmp] = false;
    };
    // whoever currently sits in the accumulator (other than `keep`) moves to a tile-sized temporary
    auto spill_acc = [&](size_t keep) {
      for (size_t i = 0; i < st.size(); ++i) {
        if (i == keep || st[i].where != Sym::ACC) continue;
        int k = -1;
        for (int t = 0; t < kFastTmps; ++t)
          if (!tmp_used[t]) { k = t; break; }
        if (k < 0) { ok = false; return; }
        tmp_used[k] = true;
        if (k + 1 > max_tmps) max_tmps = k + 1;
        femit(FO_ST_TMP, (uint8_t)k, 0, 0);
        st[i].where = Sym::TMP;
        st[i].tmp = (uint8_t)k;
      }
    };
    auto load_acc = [&](size_t i) {  // make entry i the accumulator
      if (st[i].where == Sym::ACC) return;
      spill_acc(i);
      if (st[i].where == Sym::COL) femit_load(FO_LD_COL, 2, st[i].col, map_load(st[i].load));
      else if (st[i].where == Sym::LIT) femit_load(FO_LD_LIT, 1, st[i].lit, 0);
      else {
        femit_load(FO_LD_TMP, 3, st[i].tmp, 0);
        tmp_used[st[i].tmp] = false;
      }
      st[i].where = Sym::ACC;
    };
    auto emit_binary = [&](uint8_t fb) {  // st[n-2] op st[n-1] -> accumulator
      const size_t n = st.size();
      Sym& a = st[n - 2];
      Sym& b = st[n - 1];
      uint8_t rev = 0;
      const Sym* other;
      if (a.where == Sym::ACC) other = &b;
      else if (b.where == Sym::ACC) { other = &a; rev = FB_REV; }
      else { load_acc(n - 2); other = &b; }
      if (!ok) return;
      if (other->where == Sym::COL) femit(FO_OP_COL, fb | rev, map_load(other->load), other->col);
      else if (other->where == Sym::LIT) femit(FO_OP_LIT, fb | rev, 0, other->lit);
      else femit(FO_OP_TMP, fb | rev, other->tmp, 0);
      free_sym(*other);
    };
    auto fold_lit = [&](Sym& x, i128 v) {  // constant folding of unary ops on literals
      x.lit = add_lit((uint64_t)(u128)v, (uint64_t)((u128)v >> 64));
      x.iv = iv_exact(v);
    };

    // per-thread accumulator width of fast word w in the lean kernel (the widest any of its ops needs)
    if (p.n_fast_words > (uint32_t)kLeanMaxWords) return lf_fail(__LINE__);
    for (uint32_t w = 0; w < p.n_fast_words; ++w) p.fast[w].lean_width = p.fast[w].lean_rowrel = 0;
    auto lean_word = [&](uint32_t w, uint8_t width, bool rowrel) {
      if (w >= p.n_fast_words) { ok = false; return; }
      if (p.fast[w].lean_width && (p.fast[w].lean_rowrel != 0) != rowrel) width = 8, rowrel = false;
      if (width > p.fast[w].lean_width) p.fast[w].lean_width = width;
      p.fast[w].lean_rowrel = rowrel && p.fast[w].lean_width == 4 ? 1 : 0;
    };

    const size_t n = code_.size();
    int mask_depth = 0;  // entries on the kernel's predicate-mask stack (OR / NOT trees)
    for (size_t i = 0; i < n && ok; ++i) {
      const Instr& in = code_[i];
      switch (in.op) {
        case OP_END: femit(FO_END, 0, 0, 0); break;
        case OP_PUSH_COL: {
          const ColumnMeta& c = *plan_cols_[in.a];
          // typed leaf: PUSH_COL, PRED_*, then FILTER at the top level (a conjunct: ANDed into the selection), anything else
          // inside an OR / NOT tree (pushed onto the predicate-mask stack)
          const bool is_leaf = i + 1 < select_end_ && (code_[i + 1].op == OP_PRED_I || code_[i + 1].op == OP_PRED_U || code_[i + 1].op == OP_PRED_D ||
                                                       code_[i + 1].op == OP_PRED_F || code_[i + 1].op == OP_PRED_ISNULL ||
                                                       code_[i + 1].op == OP_PRED_NOTNULL || code_[i + 1].op == OP_PRED_ALL ||
                                                       code_[i + 1].op == OP_IN_BITS || code_[i + 1].op == OP_IN_D || code_[i + 1].op == OP_IN_F);
          if (is_leaf) {
            const bool conjunct = i + 2 < n && code_[i + 2].op == OP_FILTER && mask_depth == 0;
            const Instr& pr = code_[i + 1];
            if ((pr.op == OP_PRED_F || pr.op == OP_IN_F) && c.load_kind != LK_F64 && c.load_kind != LK_F32) return lf_fail(__LINE__);
            if (!conjunct) {
              if (mask_depth >= 8) return lf_fail(__LINE__);
              ++mask_depth;
            }
            const uint32_t push = conjunct ? 0u : 1u;
            // NULL never satisfies a typed predicate: a nullable column's leaf starts from its valid rows
            if (conjunct && c.nullable && (pr.op == OP_PRED_NOTNULL || pr.op == OP_PRED_I || pr.op == OP_PRED_U || pr.op == OP_PRED_D ||
                                           pr.op == OP_PRED_F || pr.op == OP_IN_BITS || pr.op == OP_IN_D || pr.op == OP_IN_F))
              femit(FO_VALID, in.a, 0, 0);
            if (pr.op == OP_IN_BITS || pr.op == OP_IN_D || pr.op == OP_IN_F) {
              // IN list: equality of the 64-bit images (Decimal128 entries that fit i64; the others can match no narrow value)
              std::vector<Lit> run;
              for (uint32_t k = 0; k < pr.b; ++k) {
                const Lit& L = lits_[pr.c + k];
                if (pr.op == OP_IN_F) {
                  // IEEE equality on the f64 image (an f32 column is widened as it is loaded): NaN equals nothing, a zero
                  // of either sign equals both
                  double d;
                  memcpy(&d, &L.lo, 8);
                  if (d != d) continue;
                  if (d == 0.0) {
                    run.push_back(mk_lit_i((i128)0));
                    run.push_back(mk_lit_i((i128)INT64_MIN));
                  } else {
                    run.push_back(mk_lit_i((i128)(int64_t)L.lo));
                  }
                  continue;
                }
                if (pr.op == OP_IN_D) {
                  const i128 v = (i128)(((u128)L.hi << 64) | (u128)L.lo);
                  if (!fits_i64(v)) {
                    if (c.load_kind == LK_D128) return lf_fail(__LINE__);
                    continue;
                  }
                }
                run.push_back(mk_lit_i((i128)(int64_t)L.lo));
              }
              if (c.load_kind == LK_D128 && !c.dec_fits_i64) return lf_fail(__LINE__);
              if (lits_.size() + run.size() + 1 > (size_t)kMaxLits) return lf_fail(__LINE__);  // (+1: the kernel reads a (lo, hi) pair before it looks at g)
              const uint32_t first = run.empty() ? 0u : add_lit_run(run);
              femit(FO_LEAF, in.a, map_load(in.b), first);
              f.back().g = 3u;
              f.back().f = (uint32_t)run.size();
              f.back().e = push;
              i += conjunct ? 2 : 1;
              break;
            }
            if (pr.op == OP_PRED_F) {
              // floats compare by partial_cmp (NaN matches nothing, -0 == +0): as a signed range over the order-preserving
              // integer image  k(v) = bits ^ ((bits >> sign) & MAX)  of the column's own width
              const bool f32 = c.load_kind == LK_F32;
              auto key = [&](double d) -> int64_t {
                if (f32) {
                  const float x = (float)d;
                  int32_t b;
                  memcpy(&b, &x, 4);
                  return (int64_t)(b ^ ((b >> 31) & INT32_MAX));
                }
                int64_t b;
                memcpy(&b, &d, 8);
                return b ^ ((b >> 63) & INT64_MAX);
              };
              auto lit_f = [&](uint32_t idx) { double d; const uint64_t b = lits_[idx].lo; memcpy(&d, &b, 8); return d; };
              const int64_t kninf = key(-INFINITY), kpinf = key(INFINITY);
              int64_t lo = kninf, hi = kpinf;
              bool empty = false;
              const int lk = pr.a & 3, uk = (pr.a >> 2) & 3, eq = (pr.a >> 4) & 1;
              if (eq) {
                const double a = lit_f(pr.c);
                if (a != a) empty = true;
                else if (a == 0.0) { lo = -1; hi = 0; }
                else lo = hi = key(a);
              } else {
                uint32_t li = pr.c;
                if (lk != LLKV_BOUND_UNBOUNDED) {
                  const double a = lit_f(li++);
                  if (a != a) empty = true;
                  else if (lk == LLKV_BOUND_INCLUDED) lo = a == 0.0 ? -1 : key(a);
                  else if (a == INFINITY) empty = true;
                  else lo = (a == 0.0 ? 0 : key(a)) + 1;
                }
                if (uk != LLKV_BOUND_UNBOUNDED) {
                  const double b = lit_f(li);
                  if (b != b) empty = true;
                  else if (uk == LLKV_BOUND_INCLUDED) hi = b == 0.0 ? 0 : key(b);
                  else if (b == -INFINITY) empty = true;
                  else hi = (b == 0.0 ? -1 : key(b)) - 1;
                }
              }
              if (lo < kninf) lo = kninf;
              if (hi > kpinf) hi = kpinf;
              if (lo > hi) empty = true;
              std::vector<Lit> run = {mk_lit_i(empty ? 1 : lo), mk_lit_i(empty ? 0 : hi)};
              if (lits_.size() + 2 > (size_t)kMaxLits) return lf_fail(__LINE__);
              const uint32_t first = add_lit_run(run);
              femit(FO_LEAF, in.a, f32 ? (uint32_t)LKF_4 : (uint32_t)LKF_8, first);
              f.back().g = 2u;
              f.back().e = push;
              i += conjunct ? 2 : 1;
              break;
            }
            if (pr.op == OP_PRED_ALL || pr.op == OP_PRED_NOTNULL || (pr.op == OP_PRED_ISNULL && (c.nullable || push))) {
              // Range(Unbounded, Unbounded) is true on every row, IS NOT NULL on the valid ones, IS NULL on the others
              if (push) femit(FO_VALID, in.a, pr.op == OP_PRED_ALL ? 2 : pr.op == OP_PRED_ISNULL ? 1 : 0, 1);
              else if (pr.op == OP_PRED_ISNULL) femit(FO_VALID, in.a, 1, 0);
              i += conjunct ? 2 : 1;
              break;
            }
            {
              const bool uns = pr.op == OP_PRED_U;
              i128 tmin, tmax;
              if (uns) { tmin = 0; tmax = (i128)UINT64_MAX; } else { tmin = (i128)INT64_MIN; tmax = (i128)INT64_MAX; }
              // the column's own value range bounds the comparison domain (and lets 32-bit columns compare in 32 bits)
              const Iv ci = column_interval(c);
              if (ci.known) { if (ci.lo > tmin) tmin = ci.lo; if (ci.hi < tmax) tmax = ci.hi; }
              if (c.load_kind == LK_I32 || c.load_kind == LK_D32) { if (tmin < INT32_MIN) tmin = INT32_MIN; if (tmax > INT32_MAX) tmax = INT32_MAX; }
              i128 lo = tmin, hi = tmax;
              bool empty = pr.op == OP_PRED_ISNULL;
              if (!empty) {
                const int lk = pr.a & 3, uk = (pr.a >> 2) & 3, eq = (pr.a >> 4) & 1;
                auto lit_val = [&](uint32_t idx) -> i128 {
                  const Lit& L = lits_[idx];
                  if (uns) return (i128)L.lo;
                  if (pr.op == OP_PRED_D) return (i128)(((u128)L.hi << 64) | (u128)L.lo);
                  return (i128)(int64_t)L.lo;
                };
                if (eq) {
                  lo = hi = lit_val(pr.c);
                } else {
                  uint32_t li = pr.c;
                  if (lk != LLKV_BOUND_UNBOUNDED) {
                    const i128 v = lit_val(li++);
                    if (lk == LLKV_BOUND_EXCLUDED) { if (v >= tmax) empty = true; else lo = v + 1; } else lo = v;
                  }
                  if (uk != LLKV_BOUND_UNBOUNDED) {
                    const i128 v = lit_val(li);
                    if (uk == LLKV_BOUND_EXCLUDED) { if (v <= tmin) empty = true; else hi = v - 1; } else hi = v;
                  }
                }
                if (lo < tmin) lo = tmin;
                if (hi > tmax) hi = tmax;
                if (lo > hi) empty = true;
              }
              Lit a, b;
              if (empty) { a = mk_lit_i(1); b = mk_lit_i(0); }
              else { a = mk_lit_i(lo); b = mk_lit_i(hi); }
              std::vector<Lit> run = {a, b};
              if (lits_.size() + 2 > (size_t)kMaxLits) return lf_fail(__LINE__);
              const uint32_t first = add_lit_run(run);
              femit(FO_LEAF, in.a, map_load(in.b), first);
              f.back().g = uns ? 1u : 0u;
              if (c.load_kind == LK_STR8 || c.load_kind == LK_U8 || c.load_kind == LK_U64) f.back().g = 1u;
              f.back().e = push;  // (1: the leaf's masks go onto the predicate-mask stack)
              i += conjunct ? 2 : 1;
              break;
            }
          }
          Sym x;
          x.where = Sym::COL;
          x.col = in.a;
          x.load = in.b;
          x.iv = column_interval(c);
          x.nm = c.nullable ? (1u << in.a) : 0u;
          st.push_back(x);
          break;
        }
        case OP_PUSH_LIT: {
          if (in.b) return lf_fail(__LINE__);
          const Lit& L = lits_[in.c];
          const i128 v = (i128)(((u128)L.hi << 64) | (u128)L.lo);
          Sym x;
          x.where = Sym::LIT;
          x.lit = in.c;
          if (fits_i64(v)) x.iv = iv_exact(v);
          else if (L.hi == 0) x.iv = iv_exact((i128)(int64_t)L.lo);  // f64 bits / unsigned stored with hi = 0
          else return lf_fail(__LINE__);
          st.push_back(x);
          break;
        }
        case OP_POP:
          if (st.empty()) return lf_fail(__LINE__);
          free_sym(st.back());
          st.pop_back();
          break;
        case OP_ADD_I: case OP_SUB_I: case OP_MUL_I: case OP_ADD_D: case OP_SUB_D: case OP_MUL_D: {
          if (st.size() < 2) return lf_fail(__LINE__);
          const Iv b = st[st.size() - 1].iv, a = st[st.size() - 2].iv;
          const bool is_d = in.op == OP_ADD_D || in.op == OP_SUB_D || in.op == OP_MUL_D;
          const int k = (in.op == OP_ADD_I || in.op == OP_ADD_D) ? 0 : (in.op == OP_SUB_I || in.op == OP_SUB_D) ? 1 : 2;
          const Iv r = iv_arith(k, a, b);
          uint8_t fb;
          if (iv_fits_i64(r)) fb = k == 0 ? FB_ADD : k == 1 ? FB_SUB : (iv_fits_i32(a) && iv_fits_i32(b) ? FB_MUL32 : FB_MUL);
          else if (is_d) fb = k == 0 ? FB_ADD_CK : k == 1 ? FB_SUB_CK : FB_MUL_CK;  // overflow -> rerun on the 128-bit interpreter
          else return lf_fail(__LINE__);  // a real i64 overflow is an error with its own message: general interpreter
          // (a checked operation would also look at the garbage under a NULL: nullable operands keep to proven ranges)
          const uint32_t nm = st[st.size() - 1].nm | st[st.size() - 2].nm;
          if (nm && (fb == FB_ADD_CK || fb == FB_SUB_CK || fb == FB_MUL_CK)) return lf_fail(__LINE__);
          emit_binary(fb);
          st.pop_back();
          st.back().where = Sym::ACC;
          st.back().iv = iv_fits_i64(r) ? r : Iv();
          st.back().nm = nm;
          break;
        }
        case OP_ADD_F: case OP_SUB_F: case OP_MUL_F: {
          if (st.size() < 2) return lf_fail(__LINE__);
          const uint32_t nm = st[st.size() - 1].nm | st[st.size() - 2].nm;
          emit_binary(in.op == OP_ADD_F ? FB_ADD_F : in.op == OP_SUB_F ? FB_SUB_F : FB_MUL_F);
          st.pop_back();
          st.back().where = Sym::ACC;
          st.back().iv = Iv();
          st.back().iv.is_float = true;
          st.back().nm = nm;
          break;
        }
        case OP_CAST_D_DOWN: {
          if (st.empty() || !st.back().iv.known || in.a > 18) return lf_fail(__LINE__);
          const i128 d = pow10_i128(in.a);
          const Iv src = st.back().iv;
          Iv x = src;
          x.lo = round_div(x.lo, d);
          x.hi = round_div(x.hi, d);
          const i128 lim = in.b >= 39 ? ((i128)1 << 126) : pow10_i128(in.b);
          if (!(x.lo > -lim && x.hi < lim)) return lf_fail(__LINE__);  // the precision check could turn a value into NULL
          if (st.back().where == Sym::LIT) { fold_lit(st.back(), x.lo); break; }
          load_acc(st.size() - 1);
          // the 32-bit division needs the divisor in 32 bits too: 10^k for k <= 9
          femit(FO_DIVR, in.a, src.lo >= 0 ? (src.hi < ((i128)1 << 32) && in.a <= 9 ? 2 : 1) : 0, 0);
          st.back().iv = x;
          break;
        }
        case OP_CAST_I_D: case OP_CAST_D_UP: case OP_RESCALE_DX: {
          if (st.empty() || !st.back().iv.known || in.a > 18) return lf_fail(__LINE__);
          if (in.op == OP_CAST_I_D && in.c) return lf_fail(__LINE__);
          const Iv r = iv_arith(2, st.back().iv, iv_exact(pow10_i128(in.a)));
          if (!iv_fits_i64(r)) return lf_fail(__LINE__);
          if (in.op != OP_RESCALE_DX) {
            const i128 lim = in.b >= 39 ? ((i128)1 << 126) : pow10_i128(in.b);
            if (!(r.lo > -lim && r.hi < lim)) return lf_fail(__LINE__);
          }
          if (st.back().where == Sym::LIT) { fold_lit(st.back(), r.lo); break; }
          if (in.a) {
            load_acc(st.size() - 1);
            femit(FO_MULP, in.a, 0, 0);
          }
          st.back().iv = r;
          break;
        }
        case OP_CAST_I_I: {
          if (st.empty()) return lf_fail(__LINE__);
          const int bits = in.a;
          if (bits < 64 && !iv_fits(st.back().iv, -((i128)1 << (bits - 1)), ((i128)1 << (bits - 1)) - 1)) return lf_fail(__LINE__);
          break;
        }
        case OP_CAST_U_F:  // an unsigned value proven below 2^63 converts like the signed image the accumulator holds
          if (st.empty() || !iv_fits(st.back().iv, 0, (i128)INT64_MAX)) return lf_fail(__LINE__);
          [[fallthrough]];
        case OP_CAST_I_F: case OP_CAST_D_F: {
          if (st.empty()) return lf_fail(__LINE__);
          load_acc(st.size() - 1);
          if (in.op == OP_CAST_I_F || in.op == OP_CAST_U_F) femit(FO_I2F, 0, 0, 0);
          else femit(FO_D2F, 0, 0, in.c);
          st.back().iv = Iv();
          st.back().iv.is_float = true;
          break;
        }
        case OP_CMP_I: case OP_CMP_U: case OP_CMP_F: case OP_CMP_D: {
          // compute_compare over two scalar expressions: both sides are exact 64-bit images here (anything wider left the
          // lowering earlier), so the comparison is one of bit patterns; the result goes onto the predicate-mask stack
          if (i >= select_end_ || st.size() < 2 || mask_depth >= 8 || in.a > LLKV_CMP_GE) return lf_fail(__LINE__);
          const size_t n2 = st.size();
          uint32_t cmp = in.a;
          const Sym* other;
          if (st[n2 - 2].where == Sym::ACC) other = &st[n2 - 1];
          else if (st[n2 - 1].where == Sym::ACC) {  // operand cmp acc: the mirrored comparison of acc with the operand
            static const uint8_t mirrored[6] = {LLKV_CMP_EQ, LLKV_CMP_NE, LLKV_CMP_GT, LLKV_CMP_GE, LLKV_CMP_LT, LLKV_CMP_LE};
            other = &st[n2 - 2];
            cmp = mirrored[cmp];
          } else {
            load_acc(n2 - 2);
            other = &st[n2 - 1];
          }
          if (!ok) return lf_fail(__LINE__);
          const uint32_t kind = in.op == OP_CMP_U ? 1u : in.op == OP_CMP_F ? 2u : 0u;
          const uint32_t nm = st[n2 - 1].nm | st[n2 - 2].nm;
          if (other->where == Sym::COL) femit(FO_CMP, cmp | (kind << 4), 0u | (map_load(other->load) << 8), other->col);
          else if (other->where == Sym::LIT) femit(FO_CMP, cmp | (kind << 4), 1u, other->lit);
          else femit(FO_CMP, cmp | (kind << 4), 2u, other->tmp);
          f.back().h = nm;
          free_sym(st[n2 - 1]);
          free_sym(st[n2 - 2]);
          st.pop_back();
          st.pop_back();
          ++mask_depth;
          break;
        }
        case OP_ISNULL: {
          // Expr::IsNull over a scalar expression: NULL exactly where some column it depends on is NULL (data-dependent
          // NULLs — a division by zero, a failed safe cast — never reach this lowering); the result itself is never NULL
          if (i >= select_end_ || st.empty() || mask_depth >= 8) return lf_fail(__LINE__);
          const uint32_t nm = st.back().nm;
          free_sym(st.back());
          st.pop_back();
          femit(FO_ISNULL, in.a ? 1u : 0u, 0, 0);
          f.back().h = nm;
          ++mask_depth;
          break;
        }
        case OP_AND: case OP_OR:
          if (mask_depth < 2) return lf_fail(__LINE__);
          femit(in.op == OP_AND ? FO_MASK_AND : FO_MASK_OR, 0, 0, 0);
          --mask_depth;
          break;
        case OP_NOT:
          if (mask_depth < 1) return lf_fail(__LINE__);
          femit(FO_MASK_NOT, 0, 0, 0);
          break;
        case OP_BOOL_LIT:
          if (i >= select_end_ || mask_depth >= 8) return lf_fail(__LINE__);  // (also the accumulator of an IN list: not on this path)
          femit(FO_MASK_LIT, in.a ? 1u : 0u, 0, 0);
          ++mask_depth;
          break;
        case OP_FILTER:
          if (mask_depth != 1) return lf_fail(__LINE__);
          femit(FO_MASK_FILTER, 0, 0, 0);
          mask_depth = 0;
          break;
        case OP_MVCC: femit(FO_MVCC, in.a, in.b, 0); break;  // (NULL created_by / deleted_by take their defaults in the kernel)
        case OP_SELECT_DONE: femit(FO_SELECT_DONE, 0, 0, 0); break;
        case OP_GROUP: {
          const int nk = in.a;
          if ((int)st.size() < nk) return lf_fail(__LINE__);
          for (int k = nk - 1; k >= 0; --k) {
            const Sym x = st.back();
            if (x.where != Sym::COL) return lf_fail(__LINE__);
            // a NULL key value is its own group: packed keys carry a null bit per nullable key; the single wide integer
            // key (a separate NULL row) and hashed keys stay on the general interpreter
            if (x.nm && (p.single_wide_key || !p.key_nullable[k])) return lf_fail(__LINE__);
            st.pop_back();
            p.key_col[k] = x.col;
            p.key_load[k] = (uint8_t)map_load(x.load);
          }
          femit(FO_GROUP, (uint8_t)nk, 0, 0);
          break;
        }
        case OP_AGG_COUNT_STAR: femit(FO_COUNT_STAR, 0, in.b, in.c); lean_word(in.b, 4, false); break;
        case OP_AGG_FIRSTROW: femit(FO_FIRSTROW, 0, in.b, in.c); lean_word(in.b, 4, true); break;
        case OP_AGG_COUNT: case OP_AGG_SUM_I: case OP_AGG_SUM_D: case OP_AGG_FSUM: case OP_AGG_MIN_I: case OP_AGG_MAX_I:
        case OP_AGG_MIN_F: case OP_AGG_MAX_F: case OP_AGG_FIRSTVALID: case OP_AGG_FIRSTNAN: case OP_AGG_MIN_D: case OP_AGG_MAX_D: {
          if (st.empty()) return lf_fail(__LINE__);
          uint8_t a = 0;
          uint16_t op;
          bool keep = (in.a & 1) != 0;
          uint8_t width = 8;
          bool rowrel = false;
          switch (in.op) {
            case OP_AGG_MIN_D: case OP_AGG_MAX_D: {
              // Decimal128 MIN/MAX over values proven to sit strictly inside i64: the thread-private state is one
              // order-preserving u64 (its identity is then never a real value); the global state stays the 128-bit pair
              const Iv& v = st.back().iv;
              if (!v.known || !(v.lo > (i128)INT64_MIN && v.hi < (i128)INT64_MAX)) return lf_fail(__LINE__);
              op = in.op == OP_AGG_MIN_D ? FO_MIN_I : FO_MAX_I;
              a = 0x80;
              break;
            }
            case OP_AGG_COUNT: op = FO_COUNT; width = 4; break;
            case OP_AGG_SUM_I: case OP_AGG_SUM_D: {
              op = FO_SUM;
              // value class: every consumer thread keeps a private accumulator and folds at most 2^15 rows per launch
              // (kLeanRowsPerThreadLog2): values in [0, 2^16) sum exactly in 32 bits, |v| < 2^47 in 64 bits
              const Iv& v = st.back().iv;
              if (v.known) {
                i128 m = v.hi > -v.lo ? v.hi : -v.lo;
                if (m < 0) m = 0;
                if (v.lo >= 0 && m < ((i128)1 << 16)) { a = 1; width = 4; }
                else if (m < ((i128)1 << 47)) a = 2;
              }
              if (in.op == OP_AGG_SUM_D) a |= 0x80;
              break;
            }
            case OP_AGG_FSUM: op = FO_FSUM; break;
            case OP_AGG_MIN_I: op = FO_MIN_I; break;
            case OP_AGG_MAX_I: op = FO_MAX_I; break;
            case OP_AGG_MIN_F: op = FO_MIN_F; break;
            case OP_AGG_MAX_F: op = FO_MAX_F; break;
            case OP_AGG_FIRSTVALID: op = FO_FIRSTVALID; keep = true; width = 4; rowrel = true; break;
            default: op = FO_FIRSTNAN; keep = true; width = 4; rowrel = true; break;
          }
          lean_word(in.b, width, rowrel);
          if (op != FO_COUNT && op != FO_FIRSTVALID) load_acc(st.size() - 1);  // counts do not look at the value
          femit(op, a, in.b, in.c);
          f.back().h = st.back().nm;
          if (op == FO_SUM) {  // operand proven in [0, 2^32): its width in bits (packed tuples of a partitioned GROUP BY)
            const Iv& v = st.back().iv;
            if (v.known && v.lo >= 0 && v.hi < ((i128)1 << 32)) {
              uint32_t bits = 1;
              while (bits < 32 && (v.hi >> bits) != 0) ++bits;
              f.back().g = bits;
            }
          }
          if (!keep) {
            free_sym(st.back());
            st.pop_back();
          }
          break;
        }
        default: return lf_fail(-(int)in.op);  // anything else (OR/NOT trees, IN lists, float leaves, divisions, 128-bit min/max, ...)
      }
      if (f.size() >= (size_t)kMaxFastInstr) return lf_fail(__LINE__);
    }
    if (!ok) return lf_fail(__LINE__);
    p.n_finstr = (uint32_t)f.size();
    p.fast_tmps = (uint32_t)max_tmps;
    for (size_t i = 0; i < f.size(); ++i) p.fcode[i] = f[i];
    return true;
  }
};

}  // namespace

int prim_type_width(int32_t type) {
  switch (type) {
    case LLKV_PT_UINT64: case LLKV_PT_INT64: case LLKV_PT_FLOAT64: case LLKV_PT_DATE64: return 8;
    case LLKV_PT_INT32: case LLKV_PT_UINT32: case LLKV_PT_FLOAT32: case LLKV_PT_DATE32: return 4;
    case LLKV_PT_INT16: case LLKV_PT_UINT16: return 2;
    case LLKV_PT_INT8: case LLKV_PT_UINT8: case LLKV_PT_BOOLEAN: return 1;
    case LLKV_PT_DECIMAL128: return 16;
    default: return 0;
  }
}

double powi_f64(double a, int b) {
  const bool recip = b < 0;
  double r = 1;
  while (true) {
    if (b & 1) r *= a;
    b /= 2;
    if (b == 0) break;
    a *= a;
  }
  return recip ? 1 / r : r;
}

int32_t compile_plan(const CompileRequest& req, CompileResult& out) {
  out.aggs.clear();
  out.keys.clear();
  out.status = 0;
  out.error.clear();
  try {
    Emitter em(req, out);
    em.run();
  } catch (const CompileError& e) {
    out.status = e.code;
    out.error = e.msg;
    return e.code;
  }
  return 0;
}

}  // namespace llkv
