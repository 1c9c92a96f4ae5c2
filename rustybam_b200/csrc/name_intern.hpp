// name_intern.hpp — name ids of PAF records (paf.rs:62-78 as rbh::Paf::from_text restates it): ids are handed out by first
// appearance in file order, query and target names share one table, and per record the query name is interned before the
// target name.  Shared by the host reader (host/rbhost.cpp) and the device parser's host step (rbcuda.cu: rb_batch_upload_paf).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstring>

namespace rbn {

// q_name(r) / t_name(r) -> {pointer, length} of record r's names; intern(p, n) -> the name's id (adding it if new).
// Consecutive records mostly repeat their names (rows of one window run, reads of one contig): the name of the record before is
// compared first, the table only sees the changes — millions of short rows otherwise spend their time hashing.
template <class QName, class TName, class Intern>
void intern_record_names(size_t n_rec, QName q_name, TName t_name, Intern intern, uint32_t* q_id, uint32_t* t_id) {
    const char *lq = nullptr, *lt = nullptr;
    size_t lqn = 0, ltn = 0;
    uint32_t lq_id = 0, lt_id = 0;
    for (size_t r = 0; r < n_rec; r++) {
        const auto q = q_name(r);
        if (!(lq && lqn == q.second && memcmp(lq, q.first, lqn) == 0)) {
            lq_id = intern(q.first, q.second);
            lq = q.first; lqn = q.second;
        }
        const auto t = t_name(r);
        if (!(lt && ltn == t.second && memcmp(lt, t.first, ltn) == 0)) {
            lt_id = intern(t.first, t.second);
            lt = t.first; ltn = t.second;
        }
        q_id[r] = lq_id;
        t_id[r] = lt_id;
    }
}

}  // namespace rbn
