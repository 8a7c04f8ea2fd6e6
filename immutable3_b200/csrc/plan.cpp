// plan.cpp — host-side planner: the reference's per-batch predicate passes folded into one
// merged test per column.
//
// Reference behaviour being folded (SURVEY.md §3.4):
//  * every SelectIterator scans all positions of the batch and only clears bits
//    (Select.scala:36-39, 67-78, 105-116, 143-154), the And/Or tag is dropped
//    (Engine.scala:237-245)  =>  the predicate list is a conjunction, order-independent;
//  * the Double constant is narrowed first: INT column `toInt`, TINYINT column `toByte`
//    (Select.scala:65,73,103,111,141,149); comparisons are strict and signed;
//  * GT/LT/EQ on a STRING column and Match on a numeric column throw
//    "Unsupported column vector" (Select.scala:41,80,118,156); NotMatch/NoOp throw
//    "Unsupported condition" (Select.scala:22).
// A conjunction of strict signed comparisons against integers on one column is exactly one
// inclusive range [lo, hi]; a conjunction of Match lists is the intersection of the lists.
#include "plan.hpp"

#include <algorithm>
#include <climits>
#include <cstring>

#include "json_min.hpp"

namespace imm3 {

int find_col(const TableMeta& t, const char* name) {
    if (!name) return -1;
    for (size_t i = 0; i < t.cols.size(); i++)
        if (t.cols[i].name == name) return (int)i;
    return -1;
}

int build_logical_plan(const TableMeta& table, const imm3_pred* preds, int npreds, const char* const* proj_cols,
                       int nproj, int64_t limit, LogicalPlan* out) {
    if (npreds < 0 || nproj < 0 || (npreds > 0 && !preds) || (nproj > 0 && !proj_cols))
        return fail(IMM3_ERR_INVALID_ARG, "query: bad predicate/projection arrays");
    *out = LogicalPlan();
    out->table = &table;
    out->limit = limit;

    // Engine.getColumns (Engine.scala:85-106): every named column must exist (Table.scala:10-13).
    for (int i = 0; i < npreds; i++) {
        if (!preds[i].col) return fail(IMM3_ERR_INVALID_ARG, "predicate %d: column is NULL", i);
        if (find_col(table, preds[i].col) < 0)
            return fail(IMM3_ERR_NOT_FOUND, "Column %s does not exist in table %s", preds[i].col, table.name.c_str());
    }
    for (int i = 0; i < nproj; i++) {
        if (!proj_cols[i]) return fail(IMM3_ERR_INVALID_ARG, "projection %d: column is NULL", i);
        int c = find_col(table, proj_cols[i]);
        if (c < 0) return fail(IMM3_ERR_NOT_FOUND, "Column %s does not exist in table %s", proj_cols[i], table.name.c_str());
        out->proj.push_back(c);
    }
    if (nproj > kMaxProjCols) return fail(IMM3_ERR_UNSUPPORTED, "more than %d projected columns", kMaxProjCols);

    std::vector<bool> seen_match(table.cols.size(), false);
    for (int i = 0; i < npreds; i++) {
        const imm3_pred& p = preds[i];
        int ci = find_col(table, p.col);
        const ColumnMeta& c = table.cols[(size_t)ci];
        if (p.op != IMM3_OP_GT && p.op != IMM3_OP_LT && p.op != IMM3_OP_EQ && p.op != IMM3_OP_MATCH)
            return fail(IMM3_ERR_UNSUPPORTED, "Unsupported condition");  // Select.scala:22
        const bool is_match = p.op == IMM3_OP_MATCH;
        if (is_match != (c.ctype == IMM3_COL_STRING))
            return fail(IMM3_ERR_UNSUPPORTED, "Unsupported column vector");  // Select.scala:41,80,118,156
        LogicalFilter* f = nullptr;
        for (auto& g : out->filters)
            if (g.col_idx == ci) f = &g;
        if (!f) {
            out->filters.emplace_back();
            f = &out->filters.back();
            f->col_idx = ci;
            if (c.ctype == IMM3_COL_INT) { f->kind = kFilterI32Range; f->lo = INT32_MIN; f->hi = INT32_MAX; }
            else if (c.ctype == IMM3_COL_TINYINT) { f->kind = kFilterI8Range; f->lo = -128; f->hi = 127; }
            else f->kind = kFilterStrMatch;
        }
        LogicalPlan::Narrowed nw{c.name, p.op, 0, 0};
        if (is_match) {
            if (p.nstrs < 0 || (p.nstrs > 0 && !p.strs)) return fail(IMM3_ERR_INVALID_ARG, "predicate %d: bad literal list", i);
            // data(x) is a k-byte string; a literal of another length can never equal it (Select.scala:37).
            std::vector<std::string> mine;
            for (int s = 0; s < p.nstrs; s++) {
                if (!p.strs[s]) return fail(IMM3_ERR_INVALID_ARG, "predicate %d: NULL literal", i);
                std::string lit(p.strs[s]);
                if ((int)lit.size() == c.width && std::find(mine.begin(), mine.end(), lit) == mine.end()) mine.push_back(lit);
            }
            if (!seen_match[(size_t)ci]) {
                f->lits = mine;
                seen_match[(size_t)ci] = true;
            } else {
                std::vector<std::string> both;
                for (auto& s : f->lits)
                    if (std::find(mine.begin(), mine.end(), s) != mine.end()) both.push_back(s);
                f->lits = both;
            }
        } else {
            nw.ival = d2i(p.num);
            nw.bval = d2b(p.num);
            int64_t k = c.ctype == IMM3_COL_INT ? (int64_t)nw.ival : (int64_t)nw.bval;
            if (p.op == IMM3_OP_GT) f->lo = std::max(f->lo, k + 1);       // data(x) > k
            else if (p.op == IMM3_OP_LT) f->hi = std::min(f->hi, k - 1);  // data(x) < k
            else { f->lo = std::max(f->lo, k); f->hi = std::min(f->hi, k); }
        }
        out->narrowed.push_back(nw);
    }
    if ((int)out->filters.size() > kMaxFilterCols)
        return fail(IMM3_ERR_UNSUPPORTED, "predicates on more than %d distinct columns", kMaxFilterCols);
    size_t lit_bytes = 0;
    for (auto& f : out->filters) {
        if (f.kind == kFilterStrMatch) {
            if (f.lits.empty()) out->always_empty = true;
            lit_bytes += f.lits.size() * (size_t)table.cols[(size_t)f.col_idx].width;
        } else if (f.lo > f.hi) {
            out->always_empty = true;
        }
        if (table.cols[(size_t)f.col_idx].codec == IMM3_CODEC_PFOR_INT) out->uses_pfor = true;
    }
    if (lit_bytes > (size_t)kLitPoolBytes)
        return fail(IMM3_ERR_UNSUPPORTED, "Match literals need %zu bytes, limit is %d", lit_bytes, kLitPoolBytes);
    int npfor = 0;
    std::vector<int> pf;
    auto note_pfor = [&](int ci) {
        if (table.cols[(size_t)ci].codec != IMM3_CODEC_PFOR_INT) return;
        out->uses_pfor = true;
        if (std::find(pf.begin(), pf.end(), ci) == pf.end()) { pf.push_back(ci); npfor++; }
    };
    for (auto& f : out->filters) note_pfor(f.col_idx);
    for (int ci : out->proj) note_pfor(ci);
    if (npfor > kMaxPforCols) return fail(IMM3_ERR_UNSUPPORTED, "more than %d PFOR_INT columns in one query", kMaxPforCols);
    return 0;
}

std::string explain_json(const LogicalPlan& lp, const char* kernel) {
    static const char* kinds[] = {"i8_range", "i32_range", "str_match"};
    std::string s = "{\"table\":\"" + json_escape(lp.table->name) + "\",\"kernel\":\"" + kernel + "\",\"always_empty\":" +
                    (lp.always_empty ? "true" : "false") + ",\"limit\":" + std::to_string(lp.limit > 0 ? lp.limit : 0) +
                    ",\"filters\":[";
    for (size_t i = 0; i < lp.filters.size(); i++) {
        const LogicalFilter& f = lp.filters[i];
        if (i) s += ",";
        s += "{\"col\":\"" + json_escape(lp.table->cols[(size_t)f.col_idx].name) + "\",\"kind\":\"" + kinds[f.kind] + "\"";
        if (f.kind == kFilterStrMatch) {
            s += ",\"lits\":[";
            for (size_t k = 0; k < f.lits.size(); k++) s += std::string(k ? "," : "") + "\"" + json_escape(f.lits[k]) + "\"";
            s += "]";
        } else {
            s += ",\"lo\":" + std::to_string(f.lo) + ",\"hi\":" + std::to_string(f.hi);
        }
        s += "}";
    }
    s += "],\"proj\":[";
    for (size_t i = 0; i < lp.proj.size(); i++)
        s += std::string(i ? "," : "") + "\"" + json_escape(lp.table->cols[(size_t)lp.proj[i]].name) + "\"";
    s += "],\"narrowed\":[";
    for (size_t i = 0; i < lp.narrowed.size(); i++) {
        auto& n = lp.narrowed[i];
        s += std::string(i ? "," : "") + "{\"col\":\"" + json_escape(n.col) + "\",\"op\":" + std::to_string(n.op) +
             ",\"int\":" + std::to_string(n.ival) + ",\"byte\":" + std::to_string((int)n.bval) + "}";
    }
    s += "]}";
    return s;
}

}  // namespace imm3
