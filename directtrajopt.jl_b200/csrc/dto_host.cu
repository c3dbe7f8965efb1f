// Host side of libdto_b200.so: descriptor validation, the closed-form structure builder that
// replaces Evaluator(prob)'s sparse-matrix construction and O(n_vars^2) index maps
// (/root/reference/src/solvers/evaluator.jl:99-288), device residency, and the C ABI of
// include/dto_b200.h.  No torch types, no CPU compute fallback: every value comes from a kernel.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <limits>
#include <mutex>
#include <new>
#include <thread>

#include "dto_internal.h"
#include "knotfun.cuh"

static thread_local std::string g_create_error;

struct ConEntry {
    long long col_local;  // local column
    long long grow;       // global 0-based row
    long long lrow;       // local 0-based row
    long long e;          // index into the constraint's dense [j][a][i] table
    int ci;
};

// Host threads that write structural zeros into the caller's Hessian buffer while the GPU computes and the copy
// engine delivers only the value-dependent runs (see HRun).  No arithmetic happens on the host.
struct ZeroFill {
    std::vector<std::thread> workers;
    std::mutex m;
    std::condition_variable cv, cv_done;
    long long gen = 0;
    int pending = 0;
    bool stop = false;
    std::function<void(int, int)> job;  // job(part, parts): writes this part's share of the constants
    int parts = 1;

    void run_part(int part) { job(part, parts); }
    void start(int nthreads) {
        parts = std::max(1, nthreads);
        for (int t = 1; t < parts; ++t)
            workers.emplace_back([this, t] {
                long long seen = 0;
                while (true) {
                    {
                        std::unique_lock<std::mutex> lk(m);
                        cv.wait(lk, [&] { return stop || gen != seen; });
                        if (stop) return;
                        seen = gen;
                    }
                    run_part(t);
                    {
                        std::lock_guard<std::mutex> lk(m);
                        if (--pending == 0) cv_done.notify_all();
                    }
                }
            });
    }
    // the calling thread takes part 0 in finish(): the workers run while the caller enqueues GPU work
    void launch(std::function<void(int, int)> j) {
        std::lock_guard<std::mutex> lk(m);
        job = std::move(j);
        pending = parts - 1;
        ++gen;
        cv.notify_all();
    }
    void finish() {
        run_part(0);
        std::unique_lock<std::mutex> lk(m);
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    ~ZeroFill() {
        {
            std::lock_guard<std::mutex> lk(m);
            stop = true;
            cv.notify_all();
        }
        for (auto& w : workers) w.join();
    }
};

// Consecutive owned knots whose Hessian columns below l0 are structurally zero (no term of the problem touches them):
// only the tail of each knot's region crosses PCIe, as one 2-D copy per run.
struct HRun {
    int k0, cnt, l0;
};

struct dto_handle {
    std::string err;
    int device = 0;
    cudaStream_t stream = nullptr;
    DProb P;
    dto_size_info sizes_global{};  // of the WHOLE problem (one batch member)
    dto_size_info sizes_local{};
    int eval_hessian = 1;
    int sharded = 0;
    int k0 = 1, k1 = 1;
    std::vector<void*> allocs;
    // host copies of the descriptor
    std::vector<dto_integrator_desc> ints;
    std::vector<dto_objective_desc> objs;
    std::vector<dto_constraint_desc> cons;
    std::vector<std::vector<int>> obj_var_offs, obj_times, con_var_offs, con_times;
    std::vector<std::vector<int>> con_own_ti;  // owned entries per constraint
    std::vector<long long> int_goff;           // global row offset of each integrator
    std::vector<long long> con_goff;           // global row offset of each constraint (after dynamics)
    std::vector<long long> jac_colptr;         // local
    std::vector<ConEntry> con_entries;         // stored constraint Jacobian entries (owned), sorted by (col, row)
    std::vector<std::vector<unsigned char>> con_stored_all;  // per constraint: stored mask over ALL times [ti][a][i]
    std::vector<int> row_is_eq;
    int G = 0;                                             // traj.global_dim
    std::vector<std::pair<long long, long long>> hess_tail;  // (global column gi, 0-based row) of the Hessian's global columns
    // device buffers
    double *dZ = nullptr, *dmu = nullptr, *dg = nullptr, *djac = nullptr, *dhess = nullptr, *dgrad = nullptr, *dJ = nullptr,
           *dpartials = nullptr, *dviol = nullptr, *dw = nullptr, *dy = nullptr;
    int* d_row_is_eq = nullptr;
    long long *d_rows0 = nullptr, *d_cols0 = nullptr;
    // ---- links between knot-range shards (shard_link.cu): exchange windows of this shard and of its peers
    XWin* xwin = nullptr;                 // own window (device memory, exportable through CUDA IPC)
    XWin* peer_win[DTO_MAX_RANKS] = {};   // every rank's window as seen from this device (own entry = xwin)
    bool peer_ipc[DTO_MAX_RANKS] = {};    // mapping opened with cudaIpcOpenMemHandle (closed in dto_destroy)
    XWin** d_peer_win = nullptr;          // device copy of peer_win
    int link_rank = -1, link_world = 0;   // < 0: not linked
    unsigned long long epoch = 0;         // iterates uploaded since the link was made
    unsigned long long waited_epoch = 0;  // the halo of this iterate has been waited for
    unsigned long long scal_seq = 0;
    // boundary Hessian block (linear-spline tdbilinear, shard_link.cu): a shard after knot 1 receives it from its left
    // neighbour, a shard with a right neighbour pushes it; hseq counts the Hessian evaluations since the link
    long long hblk_len = 0;               // doubles of the block: sum of hs_stride over the linear-spline tdbilinear integrators
    int hs_left = 0;                      // this shard's first knot needs the block (k0 > 1 and hblk_len > 0)
    unsigned long long hseq = 0;
    bool hs_push_now = false, hs_recv_now = false;  // the evaluation being enqueued pushes / receives the block of hseq
    bool link_ipc = false;                     // linked across processes: the publish kernel also waits for the right neighbour's knot
    unsigned long long* d_scal_scratch = nullptr;  // {violation bits, arrival counter} of shard_scalars_kernel
    long long launches = 0;
    long long last_d2h_bytes = 0;
    // host-pointer path: outputs leave over PCIe while later knot ranges are still being computed
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> chunk_events;
    cudaEvent_t chunk_events_at(size_t i) {  // created on demand; nullptr on failure
        while (chunk_events.size() <= i) {
            cudaEvent_t e = nullptr;
            if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
            chunk_events.push_back(e);
        }
        return chunk_events[i];
    }
    std::vector<double> pipeline_fracs;  // cumulative interval fractions of the chunk boundaries (empty = no pipelining)
    std::vector<HRun> hess_runs;         // empty: the Hessian is delivered whole
    std::vector<std::pair<long long, long long>> hess_zero_segs;  // structural-zero prefixes of the knot regions
    // host threads that zero-fill an unregistered Hessian buffer (null: no structural-zero runs, or too few threads to
    // beat the bus)
    ZeroFill* zero_fill = nullptr;
    std::vector<std::string> variants;
    // optional device timing of the interval kernels (bench.py's roofline numerator)
    int timing = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
    size_t ev_used = 0;
    double k1_ms = 0.0;
    long long k1_count = 0;
    // ---- iterate cache (evaluator.jl:474-482: the reference copies Z once per callback; the solvers call the five
    // callbacks separately on one iterate, ipopt_solver/solver.jl:85).  The handle keeps a page-locked copy of the iterate
    // that is resident on the device; a callback whose Z equals it re-uses the upload and everything already computed.
    // Early start: the FIRST callback on a new iterate -- the objective or its gradient -- also enqueues the mu-independent
    // pass (residual, Jacobian, jets) and returns as soon as its own small result is on the host; the interval kernels then
    // run while the solver goes through its next callbacks.
    int prefetch_score = 0;        // < 0: recent early starts were thrown away (the iterate changed before g / J were read): paused
    bool async_inflight = false;   // an early-started pass may still be running on `stream`
    bool prefetch_consumed = false;
    cudaEvent_t ev_small = nullptr;  // the objective / gradient of this iterate are on the device
    double* hg_pin = nullptr;        // early start: the residual is staged here ahead of the Jacobian's last block (copy-engine FIFO)
    cudaEvent_t ev_g = nullptr;
    bool g_staged = false;
    double* hZpin = nullptr;   // [batch][n_vars_local]
    bool z_valid = false;      // dZ holds hZpin
    bool have_obj = false;     // dJ, dgrad
    bool have_g = false, have_jac = false;  // dg, djac
    bool have_jets = false;    // DInt::jets of every bilinear integrator
    bool jets_ok = false;      // every interval kernel of the problem can keep / use the jets
    long long cache_hits = 0, cache_misses = 0;
    // ---- registered outputs (dto_register_outputs): the solver's own value arrays, page-locked, structural constants
    // written once; later callbacks that are handed these pointers move only the value-dependent entries
    double *reg_jac = nullptr, *reg_hess = nullptr;
    bool reg_jac_pinned = false, reg_hess_pinned = false;  // page lock taken by this handle
    bool reg_jac_sparse = false, reg_hess_sparse = false;  // constants are in place
    int jac_skip_ok = 0;             // length of the constant head of the inner knots' Jacobian columns (0: no common layout)
    // objective / gradient kernels run beside the interval kernel on a second stream (one SM is left free for them)
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_side_fork = nullptr, ev_side = nullptr;  // knot-objective pairs on the second stream
    // linked shards: the residual of the last device-pointer evaluation is complete at ev_g_ready (before the Hessian
    // assembler): dto_shard_scalars_dev then runs beside the assembler on the second stream
    cudaEvent_t ev_g_ready = nullptr, ev_scal_done = nullptr;
    const double* g_ready_ptr = nullptr;
    const double* j_ready_ptr = nullptr;
    bool g_ready_valid = false, want_g_ready = false;
    int trace = 0;                   // DTO_B200_TRACE=1: device timeline of every host-pointer call on stderr
    bool spec_jac_inflight = false;  // a speculative delivery of the Jacobian into reg_jac is on the copy stream
    bool spec_jac_done = false;      // reg_jac holds the resident iterate's Jacobian (once the copy stream has drained)
};

#define CUDA_TRY(h, call)                                                                       \
    do {                                                                                         \
        cudaError_t _e = (call);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                       \
            return DTO_ERR_CUDA;                                                                 \
        }                                                                                        \
    } while (0)

template <class T>
static T* dev_upload(dto_handle* h, const T* src, size_t count) {
    if (count == 0) return nullptr;
    void* p = nullptr;
    if (cudaMalloc(&p, count * sizeof(T)) != cudaSuccess) return nullptr;
    h->allocs.push_back(p);
    if (src) cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice);
    else cudaMemset(p, 0, count * sizeof(T));
    return (T*)p;
}

static int fail_create(dto_handle* h, int code, const std::string& msg) {
    g_create_error = msg;
    if (h) dto_destroy(h);
    return code;
}

extern "C" int dto_abi_version(void) { return DTO_B200_ABI_VERSION; }

// ---- knot programs ------------------------------------------------------------------------------
// Compile the SSA tape of a knot program (include/dto_b200.h) into the register-machine words the device interpreter
// runs (knot_program.cuh): values no output depends on are dropped, the rest are emitted depth-first in post-order from
// the outputs (operand a's subtree, then b's), each output is written out as soon as it is complete, and slots are
// allocated by linear scan (a slot is freed at the last use of its value and handed to the next value, lowest first).
// A leaf is loaded right before each use, so sum_i v_i^2 over 128 variables needs two live slots, not 128.
// Returns DTO_OK and appends the words (constants packed after them), or an error code with the message in `msg`.
static int compile_knot_program(const dto_problem_desc* d, int index, int n_vars, int n_params, int n_out, std::vector<int4>& words,
                                 std::string& msg) {
    if (index < 0 || index >= d->n_programs || !d->programs) {
        msg = "knot program index " + std::to_string(index) + " outside 0.." + std::to_string(d->n_programs - 1);
        return DTO_ERR_INVALID;
    }
    const dto_knot_program& K = d->programs[index];
    const std::string who = "knot program " + std::to_string(index) + ": ";
    if (K.n_ops < 1 || K.n_out < 1 || !K.ops || !K.out || K.n_consts < 0 || (K.n_consts > 0 && !K.consts)) {
        msg = who + "empty tape, no outputs or missing arrays";
        return DTO_ERR_INVALID;
    }
    if (K.n_ops > DTO_MAX_PROGRAM_OPS) {
        msg = who + std::to_string(K.n_ops) + " operations, above the limit of " + std::to_string(DTO_MAX_PROGRAM_OPS) +
              " (DTO_MAX_PROGRAM_OPS)";
        return DTO_ERR_UNSUPPORTED;
    }
    if (K.n_out != n_out) {
        msg = who + std::to_string(K.n_out) + " outputs where the term has " + std::to_string(n_out);
        return DTO_ERR_INVALID;
    }
    const int n = K.n_ops;
    auto op = [&](int i, int f) { return K.ops[3 * i + f]; };
    for (int i = 0; i < n; ++i) {
        const int o = op(i, 0), a = op(i, 1), b = op(i, 2);
        bool ok;
        switch (o) {
            case DTO_OP_VAR: ok = a >= 0 && a < n_vars; break;
            case DTO_OP_PARAM: ok = a >= 0 && a < n_params; break;
            case DTO_OP_CONST: ok = a >= 0 && a < K.n_consts; break;
            case DTO_OP_ADD: case DTO_OP_SUB: case DTO_OP_MUL: case DTO_OP_DIV: ok = a >= 0 && a < i && b >= 0 && b < i; break;
            case DTO_OP_NEG: case DTO_OP_SQRT: case DTO_OP_EXP: case DTO_OP_LOG: case DTO_OP_SIN: case DTO_OP_COS: case DTO_OP_TANH:
                ok = a >= 0 && a < i;
                break;
            case DTO_OP_POWC: ok = a >= 0 && a < i && b >= 0 && b < K.n_consts; break;
            default:
                msg = who + "unknown opcode " + std::to_string(o) + " at operation " + std::to_string(i);
                return DTO_ERR_INVALID;
        }
        if (!ok) {
            msg = who + "operand out of range at operation " + std::to_string(i) +
                  " (a variable, parameter or constant index beyond the term's, or a reference to a later operation)";
            return DTO_ERR_INVALID;
        }
    }
    for (int k = 0; k < K.n_out; ++k)
        if (K.out[k] < 0 || K.out[k] >= n) {
            msg = who + "output " + std::to_string(k) + " references no operation";
            return DTO_ERR_INVALID;
        }
    auto n_operands = [&](int i) {
        const int o = op(i, 0);
        return o <= DTO_OP_CONST ? 0 : (o <= DTO_OP_DIV ? 2 : 1);  // POWC's b is a constant index
    };
    // Leaves (variables, parameters, constants) cost one load and are never kept live: a leaf operand is loaded into a
    // scratch slot right before each operation that reads it.  Only computed values occupy slots between operations --
    // an infidelity |<goal|psi>|^2 reads every variable and parameter twice, and keeping those leaves live would need
    // 4n slots.
    auto leaf = [&](int i) { return op(i, 0) <= DTO_OP_CONST; };
    // post-order emission of the computed values: entries >= 0 are operations, -1 - k writes output k
    std::vector<int> order;
    std::vector<char> seen(n, 0);
    for (int k = 0; k < K.n_out; ++k) {
        std::vector<std::pair<int, int>> stack;
        if (!leaf(K.out[k])) stack.push_back({K.out[k], 0});
        while (!stack.empty()) {
            auto& top = stack.back();
            const int i = top.first;
            if (seen[i]) {
                stack.pop_back();
                continue;
            }
            if (top.second < n_operands(i)) {
                const int c = op(i, 1 + top.second++);
                if (!leaf(c) && !seen[c]) stack.push_back({c, 0});
                continue;
            }
            seen[i] = 1;
            order.push_back(i);
            stack.pop_back();
        }
        order.push_back(-1 - k);
    }
    const int len = (int)order.size();
    std::vector<int> last(n, -1);  // position of the last use of each computed value
    for (int e = 0; e < len; ++e) {
        const int i = order[e];
        if (i < 0) last[K.out[-1 - i]] = e;
        else
            for (int q = 0; q < n_operands(i); ++q) last[op(i, 1 + q)] = e;
    }
    std::vector<int> slot(n, -1), free_slots;  // free slots in descending order: the lowest is handed out first
    int n_slots = 0;
    auto give_back = [&](int sl) {
        free_slots.push_back(sl);
        std::sort(free_slots.begin(), free_slots.end(), std::greater<int>());
    };
    auto take = [&]() {
        if (free_slots.empty()) return n_slots++;
        const int sl = free_slots.back();
        free_slots.pop_back();
        return sl;
    };
    auto load = [&](int v) {  // a leaf into a scratch slot
        const int sl = take();
        words.push_back(make_int4(op(v, 0), sl, op(v, 1), 0));
        return sl;
    };
    const size_t base = words.size();
    for (int e = 0; e < len && n_slots <= DTO_MAX_PROGRAM_SLOTS; ++e) {
        const int i = order[e];
        if (i < 0) {
            const int v = K.out[-1 - i];
            const int sl = leaf(v) ? load(v) : slot[v];
            words.push_back(make_int4(DTO_OP_OUT, -1 - i, sl, 0));
            if (leaf(v) || last[v] == e) give_back(sl);
            continue;
        }
        const int o = op(i, 0), nop = n_operands(i);
        int sl[2] = {op(i, 1), op(i, 2)};  // leaf operands of an operation are indices, POWC's b a constant index
        for (int q = 0; q < nop; ++q) {
            const int c = op(i, 1 + q);
            if (!leaf(c)) sl[q] = slot[c];
            else if (q == 1 && c == op(i, 1)) sl[1] = sl[0];  // x * x of a leaf: one load
            else sl[q] = load(c);
        }
        for (int q = 0; q < nop; ++q) {  // operands whose last use this is free their slots (each slot once)
            const int c = op(i, 1 + q);
            if (q == 1 && c == op(i, 1)) continue;
            if (leaf(c) || last[c] == e) give_back(sl[q]);
        }
        slot[i] = take();
        words.push_back(make_int4(o, slot[i], sl[0], sl[1]));
    }
    if (n_slots > DTO_MAX_PROGRAM_SLOTS) {
        words.resize(base);
        msg = who + "needs more than " + std::to_string(DTO_MAX_PROGRAM_SLOTS) +
              " live values at once, above the interpreter's limit (DTO_MAX_PROGRAM_SLOTS)";
        return DTO_ERR_UNSUPPORTED;
    }
    // constants after the words, two per int4
    const int cw = (K.n_consts + 1) / 2;
    const size_t at = words.size();
    words.resize(at + cw, make_int4(0, 0, 0, 0));
    if (K.n_consts > 0) memcpy(&words[at], K.consts, sizeof(double) * K.n_consts);
    return DTO_OK;
}

// compile and upload: the device view of program `index` for a term with n_vars variables, n_params parameters and
// n_out outputs
static int upload_knot_program(dto_handle* h, const dto_problem_desc* d, int index, int n_vars, int n_params, int n_out, DProgram& pg) {
    std::vector<int4> words;
    std::string msg;
    const int rc = compile_knot_program(d, index, n_vars, n_params, n_out, words, msg);
    if (rc != DTO_OK) return fail_create(h, rc, msg);
    const int cw = (d->programs[index].n_consts + 1) / 2;
    pg.n_code = (int)words.size() - cw;
    pg.code = dev_upload(h, words.data(), words.size());
    if (!pg.code) return fail_create(h, DTO_ERR_ALLOC, "device allocation failed (knot program)");
    return DTO_OK;
}

extern "C" const char* dto_last_error(const dto_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

extern "C" void dto_destroy(dto_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    dto_unregister_outputs(h);
    for (int r = 0; r < DTO_MAX_RANKS; ++r)
        if (h->peer_ipc[r] && h->peer_win[r]) cudaIpcCloseMemHandle(h->peer_win[r]);
    for (auto& e : h->ev_pool) {
        cudaEventDestroy(e.first);
        cudaEventDestroy(e.second);
    }
    for (void* p : h->allocs) cudaFree(p);
    for (cudaEvent_t e : h->chunk_events) cudaEventDestroy(e);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->ev_side_fork) cudaEventDestroy(h->ev_side_fork);
    if (h->ev_side) cudaEventDestroy(h->ev_side);
    if (h->ev_g_ready) cudaEventDestroy(h->ev_g_ready);
    if (h->ev_scal_done) cudaEventDestroy(h->ev_scal_done);
    if (h->ev_small) cudaEventDestroy(h->ev_small);
    if (h->ev_g) cudaEventDestroy(h->ev_g);
    if (h->hg_pin) cudaFreeHost(h->hg_pin);
    if (h->hZpin) cudaFreeHost(h->hZpin);
    delete h->zero_fill;
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}


extern "C" int dto_create(const dto_problem_desc* d, dto_handle** out) {
    if (!d || !out) return fail_create(nullptr, DTO_ERR_INVALID, "null descriptor");
    *out = nullptr;
    // version 3 descriptors (no knot programs) end before n_programs: those fields are read only at version 4
    if (d->abi_version != DTO_B200_ABI_VERSION && d->abi_version != 3) return fail_create(nullptr, DTO_ERR_INVALID, "ABI version mismatch");
    const bool with_programs = d->abi_version >= 4;
    if (with_programs && (d->n_programs < 0 || (d->n_programs > 0 && !d->programs)))
        return fail_create(nullptr, DTO_ERR_INVALID, "bad knot program table");
    if (d->N < 2 || d->z < 1 || d->batch < 1) return fail_create(nullptr, DTO_ERR_INVALID, "need N >= 2, z >= 1, batch >= 1");
    if (d->dt_off < 0 || d->dt_off >= d->z) return fail_create(nullptr, DTO_ERR_INVALID, "timestep component outside the knot");
    if (d->n_integrators < 1)
        return fail_create(nullptr, DTO_ERR_UNSUPPORTED, "at least one integrator is required (dense block Hessian structure)");
    if (d->n_integrators > DTO_MAX_INT || d->n_objectives > DTO_MAX_OBJ || d->n_constraints > DTO_MAX_CON)
        return fail_create(nullptr, DTO_ERR_UNSUPPORTED, "too many integrators / objective terms / constraints");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail_create(nullptr, DTO_ERR_CUDA, "no CUDA device: libdto_b200 has no CPU fallback");
    cudaGetLastError();  // do not inherit a stale error from an earlier, unrelated call
    dto_handle* h = new (std::nothrow) dto_handle();
    if (!h) return fail_create(nullptr, DTO_ERR_ALLOC, "out of host memory");
    if (d->device >= 0) {
        if (cudaSetDevice(d->device) != cudaSuccess) return fail_create(h, DTO_ERR_CUDA, "cudaSetDevice failed");
        h->device = d->device;
    } else {
        cudaGetDevice(&h->device);
    }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess)
        return fail_create(h, DTO_ERR_CUDA, "cudaStreamCreate failed");
    for (cudaEvent_t* e : {&h->ev_fork, &h->ev_join, &h->ev_side_fork, &h->ev_side, &h->ev_g_ready, &h->ev_scal_done, &h->ev_small, &h->ev_g})
        if (cudaEventCreateWithFlags(e, cudaEventDisableTiming) != cudaSuccess) return fail_create(h, DTO_ERR_CUDA, "cudaEventCreate failed");
    // the kernels whose shared memory grows with the shape are checked against it here, so that a shape no kernel can
    // launch is rejected at construction instead of failing at its first evaluation
    int smem_optin = 0;
    if (cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device) != cudaSuccess)
        return fail_create(h, DTO_ERR_CUDA, "cudaDeviceGetAttribute(MaxSharedMemoryPerBlockOptin) failed");
    auto smem_msg = [&](const std::string& what, size_t need) {
        return what + " needs " + std::to_string(need) + " bytes of shared memory per block, above the device's limit of " +
               std::to_string(smem_optin) + " bytes";
    };

    const int N = d->N, z = d->z;
    h->eval_hessian = d->eval_hessian;
    h->sharded = d->shard_k0 > 0;
    h->k0 = h->sharded ? d->shard_k0 : 1;
    h->k1 = h->sharded ? d->shard_k1 : N;
    if (h->k0 < 1 || h->k1 > N || h->k0 > h->k1) return fail_create(h, DTO_ERR_INVALID, "bad shard range");
    if (h->sharded && d->batch != 1) return fail_create(h, DTO_ERR_UNSUPPORTED, "knot-range shards require batch == 1");
    const int G = d->global_dim;
    if (G < 0 || G > 1024) return fail_create(h, DTO_ERR_INVALID, "global_dim outside 0..1024");
    if (G > 0 && h->sharded) return fail_create(h, DTO_ERR_UNSUPPORTED, "knot-range shards do not support global variables");
    h->G = G;

    DProb& P = h->P;
    memset(&P, 0, sizeof(P));
    P.N = N;
    P.z = z;
    P.dt_off = d->dt_off;
    P.batch = d->batch;
    P.kb = h->k0;
    P.nOwn = h->k1 - h->k0 + 1;
    P.nK = P.nOwn + (h->k1 < N ? 1 : 0);
    P.nI = P.nK - 1;
    P.kc0 = 0;
    P.kc1 = P.nK;
    P.first_has_cross = h->k0 > 1;
    P.n_int = d->n_integrators;
    P.n_obj = d->n_objectives;
    P.n_con = d->n_constraints;
    P.n_vars_local = (long long)P.nK * z + G;
    P.n_grad_local = (long long)P.nOwn * z + G;
    P.gl.G = G;

    // ---- integrators -------------------------------------------------------------------------
    long long goff = 0, loff = 0;
    int doff = 0;
    for (int i = 0; i < d->n_integrators; ++i) {
        const dto_integrator_desc& s = d->integrators[i];
        h->ints.push_back(s);
        DInt& I = P.in[i];
        I.kind = s.kind;
        I.x_off = s.x_off;
        I.n = s.x_dim;
        I.u_off = s.u_off;
        I.m = s.u_dim;
        I.t_off = s.t_off;
        I.order = s.spline_order;
        I.n_carrier = s.n_carrier;
        I.doff = doff;
        I.row_off = loff;
        I.steps = s.tdb_steps > 0 ? s.tdb_steps : 1;
        if (s.x_dim < 1 || s.x_off < 0 || s.x_off + s.x_dim > z) return fail_create(h, DTO_ERR_INVALID, "integrator state component outside the knot");
        const size_t nn = (size_t)s.x_dim * s.x_dim;
        if (s.kind == DTO_INT_BILINEAR) {
            if (s.u_dim < 0 || s.u_off < 0 || s.u_off + s.u_dim > z || !s.G) return fail_create(h, DTO_ERR_INVALID, "bilinear integrator: bad drive component or missing generators");
            const size_t per = (size_t)(s.u_dim + 1) * nn;
            const size_t cnt = s.G_batch_stride ? (size_t)s.G_batch_stride * (d->batch - 1) + per : per;
            I.G = dev_upload(h, s.G, cnt);
            I.G_stride = s.G_batch_stride;
            {
                std::vector<double> rm(cnt);
                const size_t nmat = cnt / nn;
                for (size_t q = 0; q < nmat; ++q)
                    for (int r = 0; r < s.x_dim; ++r)
                        for (int c = 0; c < s.x_dim; ++c) rm[q * nn + (size_t)r * s.x_dim + c] = s.G[q * nn + (size_t)c * s.x_dim + r];
                I.Grm = dev_upload(h, rm.data(), cnt);
                if (s.G_batch_stride == 0 && s.x_dim % 8 == 0) {  // what the persistent kernel's prologue stages
                    std::vector<double> swz(per);
                    bilinear_persistent_swizzled(s.x_dim, s.u_dim, rm.data(), swz.data());
                    I.Gsw = dev_upload(h, swz.data(), per);
                }
            }
            I.hs_stride = (s.u_dim + 1) * s.x_dim + (s.u_dim + 1) * (s.u_dim + 1);
            I.variant = bilinear_dmma_supported(s.x_dim, s.u_dim) ? DTO_VAR_DMMA : DTO_VAR_GENERIC;
            // DTO_B200_KERNEL=generic|dmma pins an older variant (A/B measurements, parity tests of every variant)
            const char* pin = getenv("DTO_B200_KERNEL");
            const bool pin_generic = pin && strcmp(pin, "generic") == 0, pin_dmma = pin && strcmp(pin, "dmma") == 0;
            const bool pin_persistent = pin && strcmp(pin, "persistent") == 0;
            if (bilinear_persistent_supported(s.x_dim, s.u_dim) && s.G_batch_stride == 0 && !pin_dmma && !pin_generic) {
                I.variant = DTO_VAR_PERSISTENT;
                I.wq = dev_upload<unsigned long long>(h, nullptr, 4);
                if (!I.wq) return fail_create(h, DTO_ERR_ALLOC, "device allocation failed (work queue)");
                // small states: eight intervals per warp, one tile per jet component (bilinear_octet.cu)
                if (bilinear_octet_supported(s.x_dim, s.u_dim) && !pin_persistent) I.variant = DTO_VAR_OCTET;
            }
            if (s.G_batch_stride != 0 && bilinear_octet_supported(s.x_dim, s.u_dim) && !pin_dmma && !pin_generic && !pin_persistent) {
                // per-problem generators at small n: the octet kernel reads each problem's fragment-ordered copy
                const size_t fd = bilinear_octet_fragment_doubles(s.x_dim, s.u_dim);
                std::vector<double> frag(fd * (size_t)d->batch);
                for (int b = 0; b < d->batch; ++b)
                    bilinear_octet_fragments(s.x_dim, s.u_dim, s.G + (size_t)b * s.G_batch_stride, frag.data() + (size_t)b * fd);
                I.bfrag = dev_upload(h, frag.data(), frag.size());
                if (!I.bfrag) return fail_create(h, DTO_ERR_ALLOC, "device allocation failed (generator fragments)");
                I.variant = DTO_VAR_OCTET;
            }
            if (pin_generic) I.variant = DTO_VAR_GENERIC;
            if (s.x_dim > 96) return fail_create(h, DTO_ERR_UNSUPPORTED, "bilinear integrator: state dimension > 96 not supported");
            if (I.variant == DTO_VAR_GENERIC) {  // one block per interval holds the generator and every jet column
                const size_t need = generic_smem_bytes(s.x_dim, s.u_dim, true, d->eval_hessian);
                if (need > (size_t)smem_optin)
                    return fail_create(h, DTO_ERR_UNSUPPORTED, smem_msg("bilinear integrator: the generic kernel at state dimension " +
                                                                        std::to_string(s.x_dim) + " with " + std::to_string(s.u_dim) +
                                                                        " drives" + (d->eval_hessian ? " and the Hessian" : ""), need));
            }
        } else if (s.kind == DTO_INT_DERIVATIVE) {
            if (s.u_dim != s.x_dim || s.u_off < 0 || s.u_off + s.u_dim > z) return fail_create(h, DTO_ERR_INVALID, "derivative integrator: derivative component must match the variable's dimension");
        } else if (s.kind == DTO_INT_TDBILINEAR) {
            if (s.u_dim < 0 || s.u_off < 0 || s.u_off + s.u_dim > z || s.t_off < 0 || s.t_off >= z || !s.G)
                return fail_create(h, DTO_ERR_INVALID, "tdbilinear integrator: bad components");
            if (!tdb_available()) return fail_create(h, DTO_ERR_UNSUPPORTED, "tdbilinear integrator kernel is not built into this library");
            if (s.spline_order != 0 && s.spline_order != 1) return fail_create(h, DTO_ERR_UNSUPPORTED, "Unsupported spline order");
            I.G = dev_upload(h, s.G, nn);
            I.A = dev_upload(h, s.A, nn * s.u_dim);
            I.B = dev_upload(h, s.B, nn * s.u_dim);
            I.omega = dev_upload(h, s.omega, s.u_dim);
            I.phi = dev_upload(h, s.phi, s.u_dim);
            I.D = dev_upload(h, s.D, nn * s.n_carrier);
            I.omega_d = dev_upload(h, s.omega_d, s.n_carrier);
            I.phi_d = dev_upload(h, s.phi_d, s.n_carrier);
            {
                // 1-norms that bound ||G(u, t)||_1 for the per-interval macro-step count (tdb_item_steps)
                auto norm1 = [&](const double* M) {
                    double best = 0.0;
                    for (int c = 0; c < s.x_dim; ++c) {
                        double sum = 0.0;
                        for (int r = 0; r < s.x_dim; ++r) sum += fabs(M[(size_t)c * s.x_dim + r]);
                        best = std::max(best, sum);
                    }
                    return best;
                };
                std::vector<double> bn((size_t)std::max(s.u_dim, 1), 0.0);
                I.tdb_gnorm = norm1(s.G);
                I.tdb_wmax = 0.0;
                {   // DTO_B200_TDB_TOL=0: eight extrapolation columns everywhere (round 1); default: sized per interval
                    const char* tl = getenv("DTO_B200_TDB_TOL");
                    I.tdb_tol = tl ? atof(tl) : 1e-14;
                }
                for (int i = 0; i < s.u_dim; ++i) {
                    bn[i] = norm1(s.A + (size_t)i * nn) + norm1(s.B + (size_t)i * nn);
                    I.tdb_wmax = std::max(I.tdb_wmax, fabs(s.omega[i]));
                }
                for (int j = 0; j < s.n_carrier; ++j) {
                    I.tdb_gnorm += norm1(s.D + (size_t)j * nn);
                    I.tdb_wmax = std::max(I.tdb_wmax, fabs(s.omega_d[j]));
                }
                I.tdb_bnorm = dev_upload(h, bn.data(), bn.size());
            }
            if (s.x_dim % 8 == 0 && s.x_dim <= 64) {
                // swizzled row-major copies for the tensor-core variant (layout of dmma_tiles.cuh)
                const int nd = s.x_dim;
                const bool swz = (nd / 8) % 2 == 0;
                auto swizzled = [&](const double* src, int count) {
                    std::vector<double> out((size_t)count * nn);
                    for (int qm = 0; qm < count; ++qm)
                        for (int r = 0; r < nd; ++r)
                            for (int c = 0; c < nd; ++c)
                                out[(size_t)qm * nn + (size_t)r * nd + (swz ? (c ^ ((r & 1) << 3)) : c)] = src[(size_t)qm * nn + (size_t)c * nd + r];
                    return out;
                };
                I.Grm = dev_upload(h, swizzled(s.G, 1).data(), nn);
                if (s.u_dim > 0) {
                    I.Asw = dev_upload(h, swizzled(s.A, s.u_dim).data(), nn * s.u_dim);
                    I.Bsw = dev_upload(h, swizzled(s.B, s.u_dim).data(), nn * s.u_dim);
                }
                if (s.n_carrier > 0) I.Dsw = dev_upload(h, swizzled(s.D, s.n_carrier).data(), nn * s.n_carrier);
                int sms = 148;
                cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
                I.tdb_scratch_ctas = 2 * sms;
                // [CTA][16 warps][accumulator, start][one tile in fragment order]
                I.tdb_scratch = dev_upload<double>(h, nullptr, (size_t)I.tdb_scratch_ctas * 16 * 2 * (nd / 8) * 64);
            }
            const int np = (s.spline_order == 1 ? 2 * s.u_dim : s.u_dim) + 2;
            I.hs_stride = np * s.x_dim + np * np;
            if (s.spline_order == 1) {
                P.any_cross = 1;
                h->hblk_len += I.hs_stride;
                if (h->k0 > 1) h->hs_left = 1;
            }
            {
                const char* pin = getenv("DTO_B200_KERNEL");
                I.variant = (I.Asw != nullptr && tdb_dmma_supported(I) && !(pin && strcmp(pin, "generic") == 0)) ? DTO_VAR_DMMA : DTO_VAR_GENERIC;
            }
            if (!tdb_fits(I, (size_t)smem_optin))
                return fail_create(h, DTO_ERR_UNSUPPORTED, "tdbilinear integrator: more than 4 drives or 4 carriers, or a state too large for the device's " +
                                                           std::to_string(smem_optin) + " bytes of shared memory per block");
            if (s.x_dim > 96) return fail_create(h, DTO_ERR_UNSUPPORTED, "tdbilinear integrator: state dimension > 96 not supported");
        } else {
            return fail_create(h, DTO_ERR_UNSUPPORTED, "unknown integrator kind");
        }
        if (I.hs_stride > 0 && d->eval_hessian) {
            // a shard whose first knot receives the previous interval's block (linear-spline tdbilinear) keeps it in a
            // leading row: the assembler reads row kl - 1 = -1
            const int lead = (s.kind == DTO_INT_TDBILINEAR && s.spline_order == 1 && h->k0 > 1) ? 1 : 0;
            I.hs = dev_upload<double>(h, nullptr, (size_t)P.batch * (std::max(P.nI, 1) + lead) * I.hs_stride);
            if (!I.hs) return fail_create(h, DTO_ERR_ALLOC, "device allocation failed (Hessian scratch)");
            I.hs += (size_t)lead * I.hs_stride;
        }
        h->int_goff.push_back(goff);
        goff += (long long)s.x_dim * (N - 1);
        loff += (long long)s.x_dim * P.nI;
        doff += s.x_dim;
        h->variants.push_back(s.kind == DTO_INT_BILINEAR ? (I.variant == DTO_VAR_OCTET ? "octet" : I.variant == DTO_VAR_PERSISTENT ? "persistent" : I.variant == DTO_VAR_DMMA ? "dmma" : "generic")
                                                         : (s.kind == DTO_INT_DERIVATIVE ? "analytic" : (I.variant == DTO_VAR_DMMA ? "gbs-dmma" : "gbs")));
    }
    P.Dsum = doff;
    const long long n_dyn_global = goff, n_dyn_local = loff;
    {
        // small-state bilinear kernel + derivative integrators: one kernel writes whole Jacobian columns
        bool any_deriv = false;
        for (int i = 0; i < P.n_int; ++i) any_deriv |= P.in[i].kind == DTO_INT_DERIVATIVE;
        if (any_deriv)
            for (int i = 0; i < P.n_int && !P.analytic_fused; ++i)
                if (P.in[i].kind == DTO_INT_BILINEAR && P.in[i].variant == DTO_VAR_OCTET) P.analytic_fused = i + 1;
    }

    // ---- objectives --------------------------------------------------------------------------
    h->obj_var_offs.resize(d->n_objectives);
    h->obj_times.resize(d->n_objectives);
    for (int i = 0; i < d->n_objectives; ++i) {
        const dto_objective_desc& s = d->objectives[i];
        h->objs.push_back(s);
        DObj& O = P.ob[i];
        O.kind = s.kind;
        O.fn = s.fn;
        O.weight = s.weight;
        O.nv = s.n_vars;
        O.nvk = s.n_vars;
        O.nt = s.n_times;
        O.np = s.n_params;
        O.D = s.D;
        if (s.kind == DTO_OBJ_MINTIME || s.kind == DTO_OBJ_NULL) continue;
        if (s.kind != DTO_OBJ_QUADREG && s.kind != DTO_OBJ_KNOT && s.kind != DTO_OBJ_LINREG && s.kind != DTO_OBJ_GLOBAL_KNOT)
            return fail_create(h, DTO_ERR_UNSUPPORTED, "unknown objective kind");
        const bool with_globals = s.kind == DTO_OBJ_GLOBAL_KNOT;
        const bool program = with_programs && s.fn == DTO_L_PROGRAM;
        if ((s.kind == DTO_OBJ_KNOT || with_globals) && !knot_lfun_known(s.fn) && !program)
            return fail_create(h, DTO_ERR_UNSUPPORTED, "knot objective function is not in the device catalogue");
        const int ngv = with_globals ? s.n_gvars : 0;
        if (s.n_vars < (with_globals ? 0 : 1) || s.n_vars + ngv > DTO_MAX_KNOTFN_VARS || (s.n_vars > 0 && !s.var_offs))
            return fail_create(h, DTO_ERR_INVALID, "objective: bad variable list");
        if (with_globals && (ngv < 1 || !s.gvar_offs)) return fail_create(h, DTO_ERR_INVALID, "global objective: missing global variable list");
        std::vector<int> all_offs(s.var_offs, s.var_offs + s.n_vars), g2l(G, -1);
        for (int v = 0; v < ngv; ++v) {
            const int go = s.gvar_offs[v];
            if (go < 0 || go >= G) return fail_create(h, DTO_ERR_INVALID, "global objective: variable outside global_data");
            if (g2l[go] >= 0) return fail_create(h, DTO_ERR_UNSUPPORTED, "global objective: repeated global variable");
            g2l[go] = s.n_vars + v;
            all_offs.push_back(go);
        }
        O.nv = s.n_vars + ngv;
        for (int v = 0; v < s.n_vars; ++v) {
            if (s.var_offs[v] < 0 || s.var_offs[v] >= z) return fail_create(h, DTO_ERR_INVALID, "objective: variable outside the knot");
            for (int v2 = 0; v2 < v; ++v2)
                if (s.var_offs[v2] == s.var_offs[v]) return fail_create(h, DTO_ERR_UNSUPPORTED, "objective: repeated variable");
        }
        std::vector<int> k2o(P.nK, -1), own, ownk;
        for (int t = 0; t < s.n_times; ++t) {
            const int k = s.times[t];
            if (k < 1 || k > N) return fail_create(h, DTO_ERR_INVALID, "objective: time index outside 1..N");
            if (k >= h->k0 && k <= h->k1) {
                if (k2o[k - h->k0] >= 0) return fail_create(h, DTO_ERR_UNSUPPORTED, "objective: repeated time index");
                k2o[k - h->k0] = (int)own.size();
                own.push_back(t);
                ownk.push_back(k - h->k0);
            }
        }
        O.var_offs = dev_upload(h, all_offs.data(), all_offs.size());
        O.g2l = with_globals ? dev_upload(h, g2l.data(), g2l.size()) : nullptr;
        O.own_ti = dev_upload(h, own.data(), own.size());
        O.own_knot = dev_upload(h, ownk.data(), ownk.size());
        O.nt_own = (int)own.size();
        O.own_kmin = ownk.empty() ? 0 : *std::min_element(ownk.begin(), ownk.end());
        O.own_kmax = ownk.empty() ? -1 : *std::max_element(ownk.begin(), ownk.end());
        O.knot_to_own = dev_upload(h, k2o.data(), k2o.size());
        if (s.kind == DTO_OBJ_QUADREG || s.kind == DTO_OBJ_LINREG) {
            if (!s.R) return fail_create(h, DTO_ERR_INVALID, "regularizer: missing R");
            for (int v = 0; v < s.n_vars; ++v)
                if (s.var_offs[v] == d->dt_off) return fail_create(h, DTO_ERR_UNSUPPORTED, "regularizer on the timestep component itself is not supported");
            O.R = dev_upload(h, s.R, s.n_vars);
            O.baseline = (s.kind == DTO_OBJ_QUADREG && s.baseline) ? dev_upload(h, s.baseline, (size_t)s.n_vars * N) : nullptr;
        } else {
            if (!s.Qs || (s.n_params > 0 && !s.params)) return fail_create(h, DTO_ERR_INVALID, "knot objective: missing Qs/params");
            O.params = dev_upload(h, s.params, (size_t)std::max(1, s.n_params) * s.n_times);
            O.Qs = dev_upload(h, s.Qs, s.n_times);
            if (program) {
                const int rc = upload_knot_program(h, d, s.program, O.nv, s.n_params, 1, O.prog);
                if (rc != DTO_OK) return rc;
            }
        }
    }

    P.hess_tab = nullptr;
    if (d->eval_hessian) {  // stream-out gather table of the Hessian assembler (assemble.cu), knots with cross rows
        const size_t need = hessian_assemble_smem_bytes(P);
        if (need > (size_t)smem_optin)
            return fail_create(h, DTO_ERR_UNSUPPORTED, smem_msg("Hessian assembly of a knot of " + std::to_string(P.z) + " variables" +
                                                                (P.any_cross ? " coupled to its neighbour" : ""), need));
        const int zz = P.z;
        std::vector<unsigned int> tab((size_t)zz * zz + (size_t)zz * (zz + 1) / 2);
        size_t e = 0;
        for (int l = 0; l < zz; ++l) {  // column l: [z cross rows | l + 1 diagonal rows]
            for (int i = 0; i < zz; ++i) tab[e++] = P.any_cross ? (unsigned int)(zz * zz + i * zz + l) : 0xFFFFFFFFu;
            for (int i = 0; i <= l; ++i) tab[e++] = (unsigned int)(i * zz + l);
        }
        P.hess_tab = dev_upload(h, tab.data(), tab.size());
    }
    {   // knot objectives: room for their Hessian pairs (assemble.cu: knot_objective_pairs_kernel)
        long long off = 0;
        for (int i = 0; i < d->n_objectives; ++i) {
            DObj& O = P.ob[i];
            O.side_off = off;
            if ((O.kind == DTO_OBJ_KNOT || O.kind == DTO_OBJ_GLOBAL_KNOT) && O.nvk > 0) off += (long long)O.nt_own * (O.nvk * (O.nvk + 1) / 2);
        }
        P.side_stride = off;
        P.knot_side = nullptr;
        if (off > 0 && d->eval_hessian) {
            P.knot_side = dev_upload<double>(h, nullptr, (size_t)off * (size_t)std::max(1, d->batch));
            if (!P.knot_side) return fail_create(h, DTO_ERR_CUDA, "out of device memory (knot objective pairs)");
        }
    }

    // ---- knot constraints ----------------------------------------------------------------------
    h->con_own_ti.resize(d->n_constraints);
    long long cgoff = 0, cloff = n_dyn_local;
    std::vector<std::vector<int>> con_own_knot(d->n_constraints);
    for (int i = 0; i < d->n_constraints; ++i) {
        const dto_constraint_desc& s = d->constraints[i];
        h->cons.push_back(s);
        const bool program = with_programs && s.fn == DTO_G_PROGRAM;
        if (!knot_cfun_known(s.fn) && !program)
            return fail_create(h, DTO_ERR_UNSUPPORTED, "knot constraint function is not in the device catalogue");
        const int ngv = s.n_gvars;
        if (ngv < 0 || s.n_vars < 0 || s.n_vars + ngv < 1 || s.n_vars + ngv > DTO_MAX_KNOTFN_VARS || s.g_dim < 1 || s.g_dim > 16 ||
            (s.n_vars > 0 && !s.var_offs) || (ngv > 0 && !s.gvar_offs))
            return fail_create(h, DTO_ERR_INVALID, "constraint: bad variable list or g_dim");
        if (s.fn == DTO_G_NORM_PRODUCT) {
            if (s.g_dim != 2 || s.n_params < 3) return fail_create(h, DTO_ERR_INVALID, "constraint: norm_product has g_dim 2 and 3 parameters");
        } else if (s.fn != DTO_G_LINEAR && !program && s.g_dim != 1)
            return fail_create(h, DTO_ERR_INVALID, "constraint: g_dim must be 1 for this function");
        std::vector<int> all_offs(s.var_offs, s.var_offs + s.n_vars), g2l(G, -1);
        for (int v = 0; v < ngv; ++v) {
            const int go = s.gvar_offs[v];
            if (go < 0 || go >= G) return fail_create(h, DTO_ERR_INVALID, "constraint: variable outside global_data");
            if (g2l[go] >= 0) return fail_create(h, DTO_ERR_UNSUPPORTED, "constraint: repeated global variable");
            g2l[go] = s.n_vars + v;
            all_offs.push_back(go);
        }
        h->con_var_offs.push_back(all_offs);
        if (!d->Z0) return fail_create(h, DTO_ERR_INVALID, "knot constraints need the initial trajectory Z0 (stored Jacobian pattern)");
        for (int v = 0; v < s.n_vars; ++v) {
            if (s.var_offs[v] < 0 || s.var_offs[v] >= z) return fail_create(h, DTO_ERR_INVALID, "constraint: variable outside the knot");
            for (int v2 = 0; v2 < v; ++v2)
                if (s.var_offs[v2] == s.var_offs[v]) return fail_create(h, DTO_ERR_UNSUPPORTED, "constraint: repeated variable");
        }
        DCon& C = P.co[i];
        C.fn = s.fn;
        C.nv = s.n_vars + ngv;
        C.nvk = s.n_vars;
        C.gd = s.g_dim;
        C.np = s.n_params;
        std::vector<int> k2o(P.nK, -1);
        for (int t = 0; t < s.n_times; ++t) {
            const int k = s.times[t];
            if (k < 1 || k > N) return fail_create(h, DTO_ERR_INVALID, "constraint: time index outside 1..N");
            if (k >= h->k0 && k <= h->k1) {
                if (k2o[k - h->k0] >= 0) return fail_create(h, DTO_ERR_UNSUPPORTED, "constraint: repeated time index");
                k2o[k - h->k0] = (int)h->con_own_ti[i].size();
                h->con_own_ti[i].push_back(t);
                con_own_knot[i].push_back(k - h->k0);
            }
        }
        C.nt_own = (int)h->con_own_ti[i].size();
        C.row_off = cloff;
        C.var_offs = dev_upload(h, all_offs.data(), all_offs.size());
        C.g2l = ngv > 0 ? dev_upload(h, g2l.data(), g2l.size()) : nullptr;
        C.own_ti = dev_upload(h, h->con_own_ti[i].data(), h->con_own_ti[i].size());
        C.own_knot = dev_upload(h, con_own_knot[i].data(), con_own_knot[i].size());
        C.knot_to_own = dev_upload(h, k2o.data(), k2o.size());
        C.params = dev_upload(h, s.params, (size_t)std::max(1, s.n_params) * s.n_times);
        if (program) {
            if (s.n_params > 0 && !s.params) return fail_create(h, DTO_ERR_INVALID, "constraint: missing params");
            const int rc = upload_knot_program(h, d, s.program, C.nv, s.n_params, s.g_dim, C.prog);
            if (rc != DTO_OK) return rc;
        }
        h->con_goff.push_back(cgoff);
        cgoff += (long long)s.g_dim * s.n_times;
        cloff += (long long)s.g_dim * C.nt_own;
    }
    const long long n_nl_global = cgoff;
    P.n_cons_local = cloff;

    // ---- stored pattern of the knot-constraint Jacobians at Z0 (problem 0) ---------------------
    // Evaluated over ALL times (a shard needs the whole pattern to know global positions) with the
    // same device templates that later produce the values.
    h->con_stored_all.resize(d->n_constraints);
    if (d->n_constraints > 0) {
        DProb Q = P;  // whole-trajectory view for the probe
        Q.batch = 1;
        Q.kb = 1;
        Q.nK = N;
        Q.nOwn = N;
        Q.nI = N - 1;
        Q.n_vars_local = (long long)N * z + G;
        Q.halo = nullptr;
        double* dZ0 = dev_upload(h, d->Z0, (size_t)N * z + G);
        long long total = 0;
        std::vector<void*> tmp;
        for (int i = 0; i < d->n_constraints; ++i) {
            const dto_constraint_desc& s = d->constraints[i];
            std::vector<int> all_ti(s.n_times), all_k(s.n_times);
            for (int t = 0; t < s.n_times; ++t) {
                all_ti[t] = t;
                all_k[t] = s.times[t] - 1;
            }
            DCon& C = Q.co[i];
            C.nt_own = s.n_times;
            C.own_ti = dev_upload(h, all_ti.data(), all_ti.size());
            C.own_knot = dev_upload(h, all_k.data(), all_k.size());
            total += (long long)s.n_times * s.g_dim * (s.n_vars + s.n_gvars);
        }
        double* dprobe = dev_upload<double>(h, nullptr, (size_t)std::max<long long>(total, 1));
        launch_constraint_pattern_probe(Q, dZ0, dprobe, h->stream, &h->launches);
        std::vector<double> probe((size_t)total);
        if (cudaMemcpyAsync(probe.data(), dprobe, sizeof(double) * total, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
            cudaStreamSynchronize(h->stream) != cudaSuccess)
            return fail_create(h, DTO_ERR_CUDA, std::string("constraint pattern probe failed: ") + cudaGetErrorString(cudaGetLastError()));
        long long off = 0;
        for (int i = 0; i < d->n_constraints; ++i) {
            const dto_constraint_desc& s = d->constraints[i];
            const long long cnt = (long long)s.n_times * s.g_dim * (s.n_vars + s.n_gvars);
            h->con_stored_all[i].resize((size_t)cnt);
            // SparseArrays' scalar setindex! does not store a zero value (either sign)
            for (long long e = 0; e < cnt; ++e) h->con_stored_all[i][(size_t)e] = probe[(size_t)(off + e)] != 0.0 ? 1 : 0;
            off += cnt;
        }
    }

    // ---- local Jacobian column pointers and constraint scatter maps ----------------------------
    // local column of variable v of constraint i at local knot kl: a knot column, or one of the G columns after them
    auto con_col = [&](int i, int v, int kl) -> size_t {
        return v < P.co[i].nvk ? (size_t)kl * z + h->con_var_offs[i][v] : (size_t)P.nK * z + h->con_var_offs[i][v];
    };
    std::vector<long long> ccount((size_t)P.nK * z + G, 0);
    for (int i = 0; i < d->n_constraints; ++i) {
        const dto_constraint_desc& s = d->constraints[i];
        const int nv = P.co[i].nv;
        for (size_t j = 0; j < h->con_own_ti[i].size(); ++j) {
            const int ti = h->con_own_ti[i][j], kl = con_own_knot[i][j];
            for (int v = 0; v < nv; ++v)
                for (int a = 0; a < s.g_dim; ++a)
                    if (h->con_stored_all[i][((size_t)ti * s.g_dim + a) * nv + v]) ccount[con_col(i, v, kl)]++;
        }
    }
    h->jac_colptr.assign((size_t)P.nK * z + G + 1, 0);
    for (int kl = 0; kl < P.nK; ++kl) {
        const long long per_col_int = (long long)P.Dsum * ((kl >= 1 ? 1 : 0) + (kl < P.nI ? 1 : 0));
        for (int l = 0; l < z; ++l) {
            const size_t c = (size_t)kl * z + l;
            h->jac_colptr[c + 1] = h->jac_colptr[c] + per_col_int + ccount[c];
        }
    }
    // global columns hold constraint entries only (integrators do not read globals: _integrators.jl:54-58)
    for (int gi = 0; gi < G; ++gi) {
        const size_t c = (size_t)P.nK * z + gi;
        h->jac_colptr[c + 1] = h->jac_colptr[c] + ccount[c];
    }
    P.nnz_jac_local = h->jac_colptr.back();
    P.jac_colptr = dev_upload(h, h->jac_colptr.data(), h->jac_colptr.size());
    P.jac_closed = h->con_entries.empty() && d->n_constraints == 0 ? 1 : 0;
    {
        std::vector<long long> fill((size_t)P.nK * z + G, 0);
        for (int i = 0; i < d->n_constraints; ++i) {
            const dto_constraint_desc& s = d->constraints[i];
            DCon& C = P.co[i];
            const int nv = C.nv;
            std::vector<long long> pos((size_t)C.nt_own * s.g_dim * nv, -1);
            for (size_t j = 0; j < h->con_own_ti[i].size(); ++j) {
                const int ti = h->con_own_ti[i][j], kl = con_own_knot[i][j];
                for (int v = 0; v < nv; ++v)
                    for (int a = 0; a < s.g_dim; ++a) {
                        if (!h->con_stored_all[i][((size_t)ti * s.g_dim + a) * nv + v]) continue;
                        const size_t c = con_col(i, v, kl);
                        const long long per_col_int = v < C.nvk ? (long long)P.Dsum * ((kl >= 1 ? 1 : 0) + (kl < P.nI ? 1 : 0)) : 0;
                        const long long e = ((long long)j * s.g_dim + a) * nv + v;
                        const long long p = h->jac_colptr[c] + per_col_int + fill[c]++;
                        pos[(size_t)e] = p;
                        ConEntry ce;
                        ce.col_local = (long long)c;
                        ce.grow = n_dyn_global + h->con_goff[i] + (long long)ti * s.g_dim + a;
                        ce.lrow = C.row_off + (long long)j * s.g_dim + a;
                        ce.e = p;  // local position
                        ce.ci = i;
                        h->con_entries.push_back(ce);
                    }
            }
            C.jac_pos = dev_upload(h, pos.data(), pos.size());
        }
        std::stable_sort(h->con_entries.begin(), h->con_entries.end(),
                         [](const ConEntry& a, const ConEntry& b) { return a.e < b.e; });
    }

    // ---- terms with global variables: slots, Hessian tail (the global columns) -----------------------
    // Pattern: objective terms mark the dense [knot vars; globals]^2 block of every listed time
    // (global_objectives.jl:268-291); constraint terms store what their Hessian at Z0 with mu = ones holds
    // (evaluator.jl:168-171, global_knot_point_constraint.jl:205-249).  Upper triangle: a global column holds the
    // coupled knot rows in ascending order, then the coupled global rows up to its own.
    if (G > 0) {
        DGlob& L = P.gl;
        std::vector<int> slot_term, slot_j, slot_kl;
        int KV = 0;
        for (int i = 0; i < d->n_objectives; ++i)
            if (P.ob[i].kind == DTO_OBJ_GLOBAL_KNOT) {
                KV = std::max(KV, P.ob[i].nvk);
                for (int t = 0; t < d->objectives[i].n_times; ++t) {  // not sharded: owned entry == position in `times`
                    slot_term.push_back(i);
                    slot_j.push_back(t);
                    slot_kl.push_back(d->objectives[i].times[t] - 1);
                }
            }
        L.S_obj = (int)slot_term.size();
        for (int i = 0; i < d->n_constraints; ++i)
            if (P.co[i].nv > P.co[i].nvk) {
                KV = std::max(KV, P.co[i].nvk);
                for (int t = 0; t < d->constraints[i].n_times; ++t) {
                    slot_term.push_back(i);
                    slot_j.push_back(t);
                    slot_kl.push_back(d->constraints[i].times[t] - 1);
                }
            }
        L.S = (int)slot_term.size();
        L.KV = KV;
        const int gtri = G * (G + 1) / 2;
        if (L.S > 0) {
            L.slot_term = dev_upload(h, slot_term.data(), slot_term.size());
            L.slot_j = dev_upload(h, slot_j.data(), slot_j.size());
            if (L.S_obj > 0) L.scratchG = dev_upload<double>(h, nullptr, (size_t)P.batch * L.S_obj * G);
            L.scratchH = dev_upload<double>(h, nullptr, (size_t)P.batch * L.S * gtri);
            if (!L.slot_term || !L.slot_j || !L.scratchH || (L.S_obj > 0 && !L.scratchG))
                return fail_create(h, DTO_ERR_ALLOC, "device allocation failed (global terms)");
        }
        std::vector<double> kg_probe((size_t)L.S * std::max(KV, 1) * G, 0.0), gg_probe;
        if (L.S > L.S_obj) {  // constraint Hessians at Z0, mu = ones, through the same device templates
            if (!d->Z0) return fail_create(h, DTO_ERR_INVALID, "constraints need the initial trajectory Z0 (stored pattern)");
            DProb Q = P;
            Q.batch = 1;
            double* dZ0 = dev_upload(h, d->Z0, (size_t)N * z + G);
            double* dprobe = dev_upload<double>(h, nullptr, kg_probe.size());
            launch_global_hessian(Q, dZ0, 1.0, nullptr, nullptr, dprobe, h->stream, &h->launches);
            gg_probe.resize((size_t)L.S * gtri);
            if (cudaMemcpyAsync(kg_probe.data(), dprobe, sizeof(double) * kg_probe.size(), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
                cudaMemcpyAsync(gg_probe.data(), L.scratchH, sizeof(double) * gg_probe.size(), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
                cudaStreamSynchronize(h->stream) != cudaSuccess)
                return fail_create(h, DTO_ERR_CUDA, std::string("global Hessian pattern probe failed: ") + cudaGetErrorString(cudaGetLastError()));
        }
        auto pair_index = [&](int gi, int gj) { return gi * G - gi * (gi - 1) / 2 + (gj - gi); };  // gi <= gj
        std::vector<std::pair<long long, long long>>& tail = h->hess_tail;
        for (int sl = 0; sl < L.S; ++sl) {
            const bool is_obj = sl < L.S_obj;
            const int ti = slot_term[sl];
            const int nvk = is_obj ? P.ob[ti].nvk : P.co[ti].nvk, nv = is_obj ? P.ob[ti].nv : P.co[ti].nv;
            const int* koffs = is_obj ? d->objectives[ti].var_offs : d->constraints[ti].var_offs;
            const int* goffs = is_obj ? d->objectives[ti].gvar_offs : d->constraints[ti].gvar_offs;
            for (int v = nvk; v < nv; ++v) {
                const int gi = goffs[v - nvk];
                for (int a = 0; a < nvk; ++a)
                    if (is_obj || kg_probe[((size_t)sl * KV + a) * G + gi] != 0.0)
                        tail.emplace_back((long long)gi, (long long)slot_kl[sl] * z + koffs[a]);
                for (int v2 = nvk; v2 < nv; ++v2) {
                    const int g2 = goffs[v2 - nvk];
                    if (g2 > gi) continue;
                    if (is_obj || gg_probe[(size_t)sl * gtri + pair_index(g2, gi)] != 0.0) tail.emplace_back((long long)gi, (long long)N * z + g2);
                }
            }
        }
        std::sort(tail.begin(), tail.end());
        tail.erase(std::unique(tail.begin(), tail.end()), tail.end());
        auto find_pos = [&](long long gi, long long row) -> long long {
            auto it = std::lower_bound(tail.begin(), tail.end(), std::make_pair(gi, row));
            return (it != tail.end() && it->first == gi && it->second == row) ? (long long)(it - tail.begin()) : -1;
        };
        std::vector<long long> kg_pos((size_t)L.S * std::max(KV, 1) * G, -1), gg_pos((size_t)gtri, -1);
        for (int sl = 0; sl < L.S; ++sl) {
            const bool is_obj = sl < L.S_obj;
            const int ti = slot_term[sl];
            const int nvk = is_obj ? P.ob[ti].nvk : P.co[ti].nvk;
            const int* koffs = is_obj ? d->objectives[ti].var_offs : d->constraints[ti].var_offs;
            for (int a = 0; a < nvk; ++a)
                for (int gi = 0; gi < G; ++gi) kg_pos[((size_t)sl * KV + a) * G + gi] = find_pos(gi, (long long)slot_kl[sl] * z + koffs[a]);
        }
        for (int gi = 0; gi < G; ++gi)
            for (int gj = gi; gj < G; ++gj) gg_pos[(size_t)pair_index(gi, gj)] = find_pos(gj, (long long)N * z + gi);
        L.kg_pos = dev_upload(h, kg_pos.data(), kg_pos.size());
        L.gg_pos = dev_upload(h, gg_pos.data(), gg_pos.size());
        L.n_hess_tail = (long long)tail.size();
    }

    // ---- sizes -----------------------------------------------------------------------------------
    const long long tri = (long long)z * (z + 1) / 2;
    P.gl.hess_tail_off = hess_knot_base(P, P.nOwn);  // base of the knot after the last owned one
    P.nnz_hess_local = P.gl.hess_tail_off + P.gl.n_hess_tail;
    h->sizes_local.n_vars = (long long)P.nOwn * z + G;
    h->sizes_local.n_dynamics_cons = n_dyn_local;
    h->sizes_local.n_nonlinear_cons = P.n_cons_local - n_dyn_local;
    h->sizes_local.n_cons = P.n_cons_local;
    h->sizes_local.nnz_jac = P.nnz_jac_local;
    h->sizes_local.nnz_hess = P.nnz_hess_local;
    h->sizes_global.n_vars = (long long)N * z + G;
    h->sizes_global.n_dynamics_cons = n_dyn_global;
    h->sizes_global.n_nonlinear_cons = n_nl_global;
    h->sizes_global.n_cons = n_dyn_global + n_nl_global;
    {
        long long stored = 0;
        for (auto& m : h->con_stored_all)
            for (unsigned char c : m) stored += c;
        h->sizes_global.nnz_jac = (long long)(N - 1) * P.Dsum * 2 * z + stored;
        h->sizes_global.nnz_hess = (long long)N * tri + (long long)(N - 1) * z * z + P.gl.n_hess_tail;
    }

    // equality flags of the local rows
    h->row_is_eq.assign((size_t)P.n_cons_local, 1);
    for (int i = 0; i < d->n_constraints; ++i)
        if (!d->constraints[i].equality)
            for (long long r = 0; r < (long long)P.co[i].nt_own * P.co[i].gd; ++r) h->row_is_eq[(size_t)(P.co[i].row_off + r)] = 0;
    h->d_row_is_eq = dev_upload(h, h->row_is_eq.data(), h->row_is_eq.size());

    // keep host copies of small arrays the structure queries need
    h->con_times.resize(d->n_constraints);
    for (int i = 0; i < d->n_constraints; ++i) {
        h->con_times[i].assign(d->constraints[i].times, d->constraints[i].times + d->constraints[i].n_times);
    }

    // ---- work buffers --------------------------------------------------------------------------
    const size_t B = (size_t)P.batch;
    h->dZ = dev_upload<double>(h, nullptr, B * (size_t)P.n_vars_local);
    h->dmu = dev_upload<double>(h, nullptr, B * (size_t)std::max<long long>(P.n_cons_local, 1));
    h->dg = dev_upload<double>(h, nullptr, B * (size_t)std::max<long long>(P.n_cons_local, 1));
    h->djac = dev_upload<double>(h, nullptr, B * (size_t)std::max<long long>(P.nnz_jac_local, 1));
    h->dgrad = dev_upload<double>(h, nullptr, B * (size_t)P.n_grad_local);
    h->dJ = dev_upload<double>(h, nullptr, B);
    h->dviol = dev_upload<double>(h, nullptr, B);
    h->dpartials = dev_upload<double>(h, nullptr, B * ((size_t)P.nOwn + (size_t)(P.nOwn + 2047) / 2048));
    if (d->eval_hessian) h->dhess = dev_upload<double>(h, nullptr, B * (size_t)std::max<long long>(P.nnz_hess_local, 1));
    if (!h->dZ || !h->dmu || !h->dg || !h->djac || !h->dgrad || !h->dJ || !h->dpartials || (d->eval_hessian && !h->dhess))
        return fail_create(h, DTO_ERR_ALLOC, "device allocation failed (work buffers)");
    {
        // iterate cache: the page-locked host copy of the resident iterate
        if (const char* tr = getenv("DTO_B200_TRACE")) h->trace = atoi(tr);
        if (cudaHostAlloc((void**)&h->hZpin, sizeof(double) * B * (size_t)P.n_vars_local, cudaHostAllocDefault) != cudaSuccess) {
            h->hZpin = nullptr;
            return fail_create(h, DTO_ERR_ALLOC, "page-locked host allocation failed (iterate cache)");
        }
        bool ok = d->eval_hessian;
        bool any = false;
        for (int i = 0; i < P.n_int; ++i) {
            if (P.in[i].kind == DTO_INT_DERIVATIVE) continue;
            any = true;
            ok = ok && P.in[i].kind == DTO_INT_BILINEAR && P.in[i].variant >= DTO_VAR_PERSISTENT;
        }
        {
            // per-interval series plans of the bilinear interval kernels (series_plan.cu); DTO_B200_SERIES_PLAN=0: size the
            // series from ||dt G(u)||_1 as round 1 did
            const char* sp = getenv("DTO_B200_SERIES_PLAN");
            if (!(sp && strcmp(sp, "0") == 0))
                for (int i = 0; i < P.n_int; ++i) {
                    DInt& I = P.in[i];
                    if (I.kind != DTO_INT_BILINEAR || I.variant < DTO_VAR_PERSISTENT) continue;
                    if (I.variant == DTO_VAR_OCTET) continue;  // n = 8 / 16: see DESIGN.md section 3
                    const dto_integrator_desc& sd = d->integrators[i];
                    if (sd.G_batch_stride != 0 || series_plan_smem(I.n, I.m) == 0) continue;  // shared sets that fit shared memory
                    std::vector<float> pm;
                    series_plan_matrices(I.n, I.m, sd.G, pm);
                    I.planmat = dev_upload(h, pm.data(), pm.size());
                    I.plan = (const double2*)dev_upload<double>(h, nullptr, 2 * B * (size_t)std::max(P.nI, 1));
                    if (!I.plan || !I.planmat) {
                        cudaGetLastError();
                        I.plan = nullptr;
                    }
                }
        }
        if (ok && any) {
            for (int i = 0; i < P.n_int && ok; ++i) {
                DInt& I = P.in[i];
                if (I.kind != DTO_INT_BILINEAR) continue;
                I.jet_stride = (I.m * (I.m + 1) / 2 + 1 + 2 * I.m) * I.n;
                I.jets = dev_upload<double>(h, nullptr, B * (size_t)std::max(P.nI, 1) * I.jet_stride);
                ok = I.jets != nullptr;
            }
            if (!ok) cudaGetLastError();
            h->jets_ok = ok;
        }
    }
    {
        // chunk boundaries of the host-pointer pipeline as cumulative fractions of the intervals.  The persistent interval
        // kernel needs many items per warp to fill the FP64 pipe (one forward item alone takes ~100 us): two ranges; the
        // octet kernel's items are small: four
        bool persistent = false;
        for (int i = 0; i < P.n_int; ++i) persistent |= P.in[i].kind == DTO_INT_BILINEAR && P.in[i].variant == DTO_VAR_PERSISTENT;
        bool tdbi = false;
        for (int i = 0; i < P.n_int; ++i) tdbi |= P.in[i].kind == DTO_INT_TDBILINEAR;
        if (tdbi) {
            // one CTA per SM works through the intervals of a range in rounds (~1 ms each at n = 64): boundaries at
            // multiples of two full rounds, so that cutting costs no partial round (c3: 296 / 592 / 888 of 999)
            int sms = 148;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
            for (int k = 2 * sms; k + sms / 2 < P.nI; k += 2 * sms) h->pipeline_fracs.push_back((k + 0.5) / (double)std::max(P.nI, 1));
        } else if (persistent) h->pipeline_fracs = {0.5};
        else h->pipeline_fracs = {0.1, 0.4, 0.7};
    }
    // ---- structural zeros of the Hessian (host-pointer path) -------------------------------------------------------
    // For bilinear/derivative problems every entry of a knot's region in a column below l0(k) is identically zero
    // (x enters the dynamics linearly: the cross block and the (x, x) block carry no term; SURVEY.md section 8a).
    // l0(k) = smallest column any term of the problem can write at knot k (column of a pair = its larger component).
    {
        bool ok = d->eval_hessian && d->batch == 1 && !P.any_cross && G == 0;
        for (int i = 0; i < P.n_int; ++i) ok = ok && (P.in[i].kind == DTO_INT_BILINEAR || P.in[i].kind == DTO_INT_DERIVATIVE);
        if (ok) {
            int l_int = z;  // knots that own an interval
            for (int i = 0; i < P.n_int; ++i) {
                const dto_integrator_desc& s = d->integrators[i];
                if (s.kind == DTO_INT_BILINEAR) {
                    for (int p = 0; p <= s.u_dim; ++p) {
                        const int c = p < s.u_dim ? s.u_off + p : d->dt_off;
                        l_int = std::min(l_int, std::max(s.x_off, c));  // (x_a, param): smallest with a = 0
                        l_int = std::min(l_int, c);                     // (param, param)
                    }
                } else {
                    l_int = std::min(l_int, std::max(s.u_off, d->dt_off));  // (xdot_a, dt)
                }
            }
            std::vector<int> l0((size_t)P.nOwn, z);
            for (int kl = 0; kl < P.nOwn; ++kl)
                if (kl < P.nI) l0[kl] = l_int;
            auto touch = [&](const int* times, int nt, int lmin) {
                for (int t = 0; t < nt; ++t) {
                    const int k = times[t];
                    if (k >= h->k0 && k <= h->k1) l0[k - h->k0] = std::min(l0[k - h->k0], lmin);
                }
            };
            for (int i = 0; i < d->n_objectives; ++i) {
                const dto_objective_desc& s = d->objectives[i];
                if (s.kind == DTO_OBJ_MINTIME || s.kind == DTO_OBJ_NULL) continue;
                int lmin = z;
                for (int v = 0; v < s.n_vars; ++v) lmin = std::min(lmin, s.var_offs[v]);
                if (s.kind == DTO_OBJ_QUADREG || s.kind == DTO_OBJ_LINREG) lmin = std::min(lmin, d->dt_off);
                touch(s.times, s.n_times, lmin);
            }
            for (int i = 0; i < d->n_constraints; ++i) {
                const dto_constraint_desc& s = d->constraints[i];
                int lmin = z;
                for (int v = 0; v < s.n_vars; ++v) lmin = std::min(lmin, s.var_offs[v]);
                touch(s.times, s.n_times, lmin);
            }
            long long zeros = 0;
            for (int kl = 0; kl < P.nOwn; ++kl) {
                const long long nc = hess_knot_has_cross(P, kl) ? z : 0;
                const long long skip = (long long)l0[kl] * nc + (long long)l0[kl] * (l0[kl] + 1) / 2;
                if (skip > 0) h->hess_zero_segs.emplace_back(hess_knot_base(P, kl), skip);
                zeros += skip;
                if (!h->hess_runs.empty() && h->hess_runs.back().l0 == l0[kl] &&
                    hess_knot_has_cross(P, h->hess_runs.back().k0) == hess_knot_has_cross(P, kl))
                    h->hess_runs.back().cnt++;
                else
                    h->hess_runs.push_back(HRun{kl, 1, l0[kl]});
            }
            // worth it only when most of the array is structural and the runs are long (few copies)
            // host threads for the zero fill: at most 4, at most half the cores; with fewer than 3 the fill would be slower
            // than the bus it relieves (one thread writes ~10 GB/s), so the whole array is delivered instead
            int nth = (int)std::min<unsigned>(4, std::max(1u, std::thread::hardware_concurrency() / 2));
            if (const char* e2 = getenv("DTO_B200_HOST_THREADS")) nth = std::max(1, std::min(32, atoi(e2)));
            if (zeros * 2 < P.nnz_hess_local || h->hess_runs.size() > 64) {
                h->hess_runs.clear();
                h->hess_zero_segs.clear();
            } else if (nth >= 3) {  // unregistered buffers need the fill threads; registered ones have their zeros in place
                h->zero_fill = new (std::nothrow) ZeroFill();
                if (h->zero_fill) h->zero_fill->start(nth);
            }
        }
    }
    {
        // Jacobian: d r_{k-1} / d z_k of a bilinear or derivative integrator is the constant [0 .. I .. 0] block
        // (bilinear_integrator.jl:81, derivative_integrator.jl:45: x_{k+1} enters linearly).  With one column layout for
        // all inner knots (no knot-constraint rows) the rest of every column is one strided copy.  Only registered Jacobian
        // arrays (dto_register_outputs) skip the heads: they get them once; an unregistered buffer would need them written
        // on every call (74 000 small memsets at c2).
        const int k0i = P.in[0].kind;
        const long long L = 2LL * P.Dsum, d1 = P.in[0].n;
        if (d->batch == 1 && P.jac_closed && G == 0 && P.nI >= 3 && (k0i == DTO_INT_BILINEAR || k0i == DTO_INT_DERIVATIVE) && 8 * (L - d1) >= 256)
            h->jac_skip_ok = (int)d1;
    }
    if (cudaStreamSynchronize(h->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess)
        return fail_create(h, DTO_ERR_CUDA, "CUDA failure during construction");
    *out = h;
    return DTO_OK;
}

extern "C" int dto_sizes(const dto_handle* h, dto_size_info* out) {
    if (!h || !out) return DTO_ERR_INVALID;
    *out = h->sharded ? h->sizes_local : h->sizes_global;
    return DTO_OK;
}

extern "C" void* dto_stream(const dto_handle* h) { return h ? (void*)h->stream : nullptr; }
extern "C" int64_t dto_launch_count(const dto_handle* h) { return h ? h->launches : 0; }
extern "C" int64_t dto_last_download_bytes(const dto_handle* h) { return h ? h->last_d2h_bytes : 0; }
extern "C" const char* dto_kernel_variant(const dto_handle* h, int i) {
    if (!h || i < 0 || i >= (int)h->variants.size()) return "";
    return h->variants[i].c_str();
}

// ---- structures -----------------------------------------------------------------------------------
// Jacobian: column-major over the local columns; inside a column [I1 prev | I1 own | I2 prev | ...]
// then the stored knot-constraint rows (evaluator.jl:119-144; SURVEY.md section 8a structure contract).
extern "C" int dto_jac_structure(const dto_handle* h, int64_t* rows, int64_t* cols) {
    if (!h || !rows || !cols) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    const int z = P.z;
    long long w = 0;
    size_t ce = 0;
    for (int kl = 0; kl < P.nK; ++kl) {
        const long long kg = (long long)P.kb - 1 + kl;  // global 0-based knot
        for (int l = 0; l < z; ++l) {
            const long long gcol = kg * z + l + 1;
            for (int i = 0; i < P.n_int; ++i) {
                const int dd = P.in[i].n;
                if (kl >= 1)
                    for (int a = 0; a < dd; ++a, ++w) {
                        rows[w] = h->int_goff[i] + (kg - 1) * dd + a + 1;
                        cols[w] = gcol;
                    }
                if (kl < P.nI)
                    for (int a = 0; a < dd; ++a, ++w) {
                        rows[w] = h->int_goff[i] + kg * dd + a + 1;
                        cols[w] = gcol;
                    }
            }
            while (ce < h->con_entries.size() && h->con_entries[ce].col_local == (long long)kl * z + l) {
                rows[w] = h->con_entries[ce].grow + 1;
                cols[w] = gcol;
                ++w;
                ++ce;
            }
        }
    }
    for (int gi = 0; gi < h->G; ++gi)  // global columns: constraint rows only
        while (ce < h->con_entries.size() && h->con_entries[ce].col_local == (long long)P.nK * z + gi) {
            rows[w] = h->con_entries[ce].grow + 1;
            cols[w] = (long long)P.N * z + gi + 1;
            ++w;
            ++ce;
        }
    return w == P.nnz_jac_local ? DTO_OK : DTO_ERR_INVALID;
}

// Hessian: upper triangle, column-major: column (k,l) holds the z rows of knot k-1 (k >= 2) and rows
// 1..l of knot k (evaluator.jl:151-203, _integrators.jl:68-77).
extern "C" int dto_hess_structure(const dto_handle* h, int64_t* rows, int64_t* cols) {
    if (!h || !rows || !cols) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    const int z = P.z;
    long long w = 0;
    for (int kl = 0; kl < P.nOwn; ++kl) {
        const long long kg = (long long)P.kb - 1 + kl;
        for (int l = 0; l < z; ++l) {
            const long long gcol = kg * z + l + 1;
            if (kg >= 1)
                for (int i = 0; i < z; ++i, ++w) {
                    rows[w] = (kg - 1) * z + i + 1;
                    cols[w] = gcol;
                }
            for (int i = 0; i <= l; ++i, ++w) {
                rows[w] = kg * z + i + 1;
                cols[w] = gcol;
            }
        }
    }
    for (const auto& e : h->hess_tail) {  // global columns
        rows[w] = e.second + 1;
        cols[w] = (long long)P.N * z + e.first + 1;
        ++w;
    }
    return w == P.nnz_hess_local ? DTO_OK : DTO_ERR_INVALID;
}

extern "C" int dto_shard_info(const dto_handle* h, dto_shard_layout* out) {
    if (!h || !out) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    out->z_begin = (long long)(P.kb - 1) * P.z;
    out->z_end = out->z_begin + (long long)P.nOwn * P.z;
    out->z_halo_end = out->z_begin + (long long)P.nK * P.z;
    out->n_local_cons = P.n_cons_local;
    out->n_local_jac = P.nnz_jac_local;
    out->n_local_hess = P.nnz_hess_local;
    return DTO_OK;
}

extern "C" int dto_shard_maps(const dto_handle* h, int64_t* con_rows, int64_t* jac_pos, int64_t* hess_pos) {
    if (!h) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    const int z = P.z, N = P.N;
    if (con_rows) {
        long long w = 0;
        for (int i = 0; i < P.n_int; ++i)
            for (int kl = 0; kl < P.nI; ++kl)
                for (int a = 0; a < P.in[i].n; ++a) con_rows[w++] = h->int_goff[i] + ((long long)P.kb - 1 + kl) * P.in[i].n + a;
        for (size_t i = 0; i < h->cons.size(); ++i)
            for (int ti : h->con_own_ti[i])
                for (int a = 0; a < h->cons[i].g_dim; ++a)
                    con_rows[w++] = h->sizes_global.n_dynamics_cons + h->con_goff[i] + (long long)ti * h->cons[i].g_dim + a;
    }
    if (jac_pos) {
        // global column pointers from the all-times stored pattern
        std::vector<long long> gcount((size_t)N * z, 0);
        for (size_t i = 0; i < h->cons.size(); ++i) {
            const dto_constraint_desc& s = h->cons[i];
            for (int t = 0; t < s.n_times; ++t)
                for (int v = 0; v < s.n_vars; ++v)
                    for (int a = 0; a < s.g_dim; ++a)
                        if (h->con_stored_all[i][((size_t)t * s.g_dim + a) * s.n_vars + v])
                            gcount[(size_t)(h->con_times[i][t] - 1) * z + h->con_var_offs[i][v]]++;
        }
        std::vector<long long> gptr((size_t)N * z + 1, 0);
        for (int k = 0; k < N; ++k) {
            const long long per = (long long)P.Dsum * ((k >= 1 ? 1 : 0) + (k < N - 1 ? 1 : 0));
            for (int l = 0; l < z; ++l) gptr[(size_t)k * z + l + 1] = gptr[(size_t)k * z + l] + per + gcount[(size_t)k * z + l];
        }
        long long w = 0;
        size_t ce = 0;
        for (int kl = 0; kl < P.nK; ++kl) {
            const long long kg = (long long)P.kb - 1 + kl;
            for (int l = 0; l < z; ++l) {
                const long long base = gptr[(size_t)kg * z + l];
                const bool gprev = kg >= 1, gown = kg < N - 1;
                for (int i = 0; i < P.n_int; ++i) {
                    const int dd = P.in[i].n, doff = P.in[i].doff;
                    const long long prev_start = base + ((gprev && gown) ? 2LL * doff : doff);
                    const long long own_start = base + ((gprev && gown) ? 2LL * doff + dd : doff);
                    if (kl >= 1)
                        for (int a = 0; a < dd; ++a) jac_pos[w++] = prev_start + a;
                    if (kl < P.nI)
                        for (int a = 0; a < dd; ++a) jac_pos[w++] = own_start + a;
                }
                const long long per = (long long)P.Dsum * ((gprev ? 1 : 0) + (gown ? 1 : 0));
                long long r = 0;
                while (ce < h->con_entries.size() && h->con_entries[ce].col_local == (long long)kl * z + l) {
                    jac_pos[w++] = base + per + r++;
                    ++ce;
                }
            }
        }
    }
    if (hess_pos) {
        const long long tri = (long long)z * (z + 1) / 2;
        long long w = 0;
        for (int kl = 0; kl < P.nOwn; ++kl) {
            const long long kg = (long long)P.kb - 1 + kl;
            const long long base = kg == 0 ? 0 : tri + (kg - 1) * ((long long)z * z + tri);
            const long long cnt = kg == 0 ? tri : (long long)z * z + tri;
            for (long long e = 0; e < cnt; ++e) hess_pos[w++] = base + e;
        }
    }
    return DTO_OK;
}

extern "C" int dto_constraint_bounds(const dto_handle* h, double* lower, double* upper) {
    if (!h || !lower || !upper) return DTO_ERR_INVALID;
    for (long long r = 0; r < h->P.n_cons_local; ++r) {
        upper[r] = 0.0;
        lower[r] = h->row_is_eq[(size_t)r] ? 0.0 : -std::numeric_limits<double>::infinity();
    }
    return DTO_OK;
}

// ---- evaluation ------------------------------------------------------------------------------------
// Knot constraints and objective: independent of the interval kernels, cheap, whole trajectory at once.
static void eval_prologue(dto_handle* h, const DProb& P, const double* dZ, double* dJ, double* dgrad, double* dg, double* djac,
                          EvalFlags f) {
    if (f.want_g || f.want_jac) launch_constraints(P, dZ, dg, djac, f, h->stream, &h->launches);
    if (dJ || dgrad) launch_objective(P, dZ, dJ, dgrad, h->dpartials, h->stream, &h->launches);
    if (dgrad) launch_global_gradient(P, dZ, dgrad, h->stream, &h->launches);
}

// The boundary block's rows, one per linear-spline tdbilinear integrator: the last local interval's (pushed to the right
// neighbour) or the leading row the left neighbour's block is received into
static HsRows hs_rows(const DProb& P, bool leading) {
    HsRows r{};
    for (int i = 0; i < P.n_int; ++i) {
        const DInt& I = P.in[i];
        if (I.kind != DTO_INT_TDBILINEAR || I.order != 1) continue;
        r.row[r.n] = I.hs + (leading ? -1LL : (long long)P.nI - 1) * I.hs_stride;
        r.len[r.n++] = I.hs_stride;
    }
    return r;
}

// Interval kernels, analytic integrators and the Hessian assembler over the active knot range of P.
static int eval_range(dto_handle* h, const DProb& P, const double* dZ, double sigma, const double* dmu, double* dg, double* djac,
                      double* dhess, EvalFlags f) {
    if (!(f.want_g || f.want_jac || f.want_hess)) return DTO_OK;
    bool fused_missed = false;
    // knot-objective Hessian pairs: they depend on Z only, so they run beside the interval kernels (second stream) and the
    // assembler below waits for them
    bool side_on_aux = false;
    if (f.want_hess && sigma != 0.0 && P.knot_side != nullptr) {
        if (P.nI >= 256) {
            CUDA_TRY(h, cudaEventRecord(h->ev_side_fork, h->stream));
            CUDA_TRY(h, cudaStreamWaitEvent(h->aux_stream, h->ev_side_fork, 0));
            side_on_aux = launch_knot_objective_pairs(P, dZ, h->aux_stream, &h->launches);
            if (side_on_aux) CUDA_TRY(h, cudaEventRecord(h->ev_side, h->aux_stream));
        } else {
            launch_knot_objective_pairs(P, dZ, h->stream, &h->launches);
        }
    }
    for (int i = 0; i < P.n_int; ++i) {
        if (P.in[i].kind == DTO_INT_DERIVATIVE) continue;
        const bool timed = h->timing && h->ev_used < h->ev_pool.size();
        if (timed) cudaEventRecord(h->ev_pool[h->ev_used].first, h->stream);
        if (P.in[i].kind == DTO_INT_BILINEAR) {
            bool done = false;
            if (P.in[i].variant == DTO_VAR_OCTET) {
                done = launch_bilinear_octet(P, i, dZ, dmu, dg, djac, f, h->stream, &h->launches);
                if (!done && P.analytic_fused == i + 1) fused_missed = true;
            }
            if (!done && P.in[i].variant >= DTO_VAR_PERSISTENT && P.in[i].G_stride == 0) done = launch_bilinear_persistent(P, i, dZ, dmu, dg, djac, f, h->stream, &h->launches);
            if (!done && f.jets != DTO_JETS_NONE) {
                h->err = "interval kernel cannot keep the forward jets between callbacks (internal)";
                return DTO_ERR_CUDA;
            }
            if (!done && P.in[i].variant >= DTO_VAR_DMMA && bilinear_dmma_supported(P.in[i].n, P.in[i].m))
                done = launch_bilinear_dmma(P, i, dZ, dmu, dg, djac, f, h->stream, &h->launches);
            if (!done) launch_bilinear_generic(P, i, dZ, dmu, dg, djac, f, h->stream, &h->launches);
            if (f.jets == DTO_JETS_USE) launch_hpp_contract(P, i, dmu, h->stream, &h->launches);
        } else if (P.in[i].kind == DTO_INT_TDBILINEAR) {
            bool done = false;
            if (P.in[i].variant == DTO_VAR_DMMA) done = launch_tdb_dmma(P, i, dZ, dmu, dg, djac, f, h->stream, &h->launches);
            if (!done) launch_tdb(P, i, dZ, dmu, dg, djac, f, h->stream, &h->launches);
        }
        if (timed) cudaEventRecord(h->ev_pool[h->ev_used++].second, h->stream);
    }
    // the last local interval's second derivatives are written: on their way to the right neighbour, which assembles the
    // knot they belong to
    if (f.want_hess && h->hs_push_now && P.nI - 1 >= P.kc0 && P.nI - 1 < P.kc1)
        launch_hs_push(h->xwin, h->peer_win[h->link_rank + 1], hs_rows(P, false), P.z, h->hblk_len, h->hseq, h->stream, &h->launches);
    if (f.want_g || f.want_jac) {
        if (fused_missed) {
            DProb Pn = P;
            Pn.analytic_fused = 0;
            launch_analytic(Pn, dZ, dg, djac, f, h->stream, &h->launches);
        } else {
            launch_analytic(P, dZ, dg, djac, f, h->stream, &h->launches);
        }
    }
    if (side_on_aux) CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_side, 0));
    if (h->want_g_ready) CUDA_TRY(h, cudaEventRecord(h->ev_g_ready, h->stream));  // every residual row is written
    if (f.want_hess && h->hs_recv_now) {
        // the first knot waits for the left neighbour's block: it is assembled in its own launch after every other knot (the
        // last range), so that the wait never holds up the rest of this shard's Hessian
        DProb Pa = P;
        Pa.kc0 = std::max(P.kc0, 1);
        launch_hessian_assemble(Pa, dZ, sigma, dmu, dhess, h->stream, &h->launches);
        if (P.kc1 >= P.nK) {
            launch_hs_receive(h->xwin, h->peer_win[h->link_rank - 1], hs_rows(P, true), P.z, h->hblk_len, h->hseq, h->stream, &h->launches);
            Pa.kc0 = 0;
            Pa.kc1 = 1;
            launch_hessian_assemble(Pa, dZ, sigma, dmu, dhess, h->stream, &h->launches, true);
        }
        return DTO_OK;  // knot-range shards have no global variables
    }
    if (f.want_hess) launch_hessian_assemble(P, dZ, sigma, dmu, dhess, h->stream, &h->launches);
    if (f.want_hess) launch_global_hessian(P, dZ, sigma, dmu, dhess, nullptr, h->stream, &h->launches);
    return DTO_OK;
}

// Series plans of the iterate in dZ (whole local trajectory), before the first interval kernel that reads them
static void launch_plans(dto_handle* h, const DProb& P, const double* dZ) {
    for (int i = 0; i < P.n_int; ++i)
        if (P.in[i].kind == DTO_INT_BILINEAR && P.in[i].plan != nullptr) launch_series_plan(P, i, dZ, h->stream, &h->launches);
}

static int check_eval_args(dto_handle* h, const double* dmu, const double* dhess) {
    if (dhess && !h->eval_hessian) {
        h->err = "evaluator was created with eval_hessian = false";
        return DTO_ERR_INVALID;
    }
    if (dhess && !dmu) {
        h->err = "Hessian evaluation needs mu";
        return DTO_ERR_INVALID;
    }
    if (dhess && h->hs_left && h->link_rank < 1) {
        h->err = "Hessian of a knot-range shard that starts after knot 1 with a linear-spline time-dependent bilinear integrator: "
                 "its first knot's block needs the left neighbour's last interval, so the shards must be linked "
                 "(dto_shard_link / dto_shard_link_local)";
        return DTO_ERR_INVALID;
    }
    return DTO_OK;
}

// A Hessian evaluation of a linked shard with a boundary block: its sequence number, and whether it pushes the block to the
// right neighbour and receives one from the left
static void begin_hs_exchange(dto_handle* h, bool hess) {
    h->hs_push_now = h->hs_recv_now = false;
    if (!hess || h->hblk_len == 0 || h->link_rank < 0) return;
    h->hs_recv_now = h->hs_left && h->link_rank > 0;
    h->hs_push_now = h->link_rank + 1 < h->link_world;
    if (h->hs_recv_now || h->hs_push_now) ++h->hseq;
}

static int prepare_halo(dto_handle* h);
static int check_link_errors(dto_handle* h);

static int run_eval(dto_handle* h, const double* dZ, double sigma, const double* dmu, double* dJ, double* dgrad, double* dg,
                    double* djac, double* dhess) {
    int rc = check_eval_args(h, dmu, dhess);
    if (rc != DTO_OK) return rc;
    h->g_ready_valid = false;
    if ((rc = prepare_halo(h)) != DTO_OK) return rc;
    begin_hs_exchange(h, dhess != nullptr);
    const DProb& P = h->P;
    EvalFlags f{dg != nullptr, djac != nullptr, dhess != nullptr};
    // The objective / gradient kernels are independent of the interval kernels and tiny (launch- and latency-bound): they run
    // on a second stream BESIDE the interval kernel, which leaves one SM free for them (0.7 % of its throughput against
    // ~17 us of serial kernels at c2).
    const bool overlap = (dJ || dgrad) && (f.want_g || f.want_jac || f.want_hess) && P.nI >= 256;
    if (overlap) {
        // forked BEFORE the series plans: the objective kernels then run beside the plan kernel and are gone when the
        // interval kernel wants its SMs (forked after it, they raced the interval kernel for them: up to 10 us)
        CUDA_TRY(h, cudaEventRecord(h->ev_fork, h->stream));  // Z (and whatever the caller enqueued before) is ready
        CUDA_TRY(h, cudaStreamWaitEvent(h->aux_stream, h->ev_fork, 0));
        launch_objective(P, dZ, dJ, dgrad, h->dpartials, h->aux_stream, &h->launches);
        if (dgrad) launch_global_gradient(P, dZ, dgrad, h->aux_stream, &h->launches);
        CUDA_TRY(h, cudaEventRecord(h->ev_join, h->aux_stream));
    }
    if (f.want_g || f.want_jac || f.want_hess) launch_plans(h, P, dZ);
    if (overlap) {
        DProb Pr = P;
        Pr.reserve_sms = 1;
        eval_prologue(h, P, dZ, nullptr, nullptr, dg, djac, f);  // knot constraints: their own rows and entries, nothing the interval kernels touch
        h->want_g_ready = h->link_rank >= 0 && dg != nullptr && dJ != nullptr && dhess != nullptr;
        rc = eval_range(h, Pr, dZ, sigma, dmu, dg, djac, dhess, f);
        const bool recorded = h->want_g_ready;
        h->want_g_ready = false;
        if (rc != DTO_OK) return rc;
        CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_join, 0));
        if (recorded) {
            h->g_ready_valid = true;
            h->g_ready_ptr = dg;
            h->j_ready_ptr = dJ;
        }
    } else {
        rc = eval_range(h, P, dZ, sigma, dmu, dg, djac, dhess, f);
        if (rc != DTO_OK) return rc;
        eval_prologue(h, P, dZ, dJ, dgrad, dg, djac, f);
    }
    CUDA_TRY(h, cudaGetLastError());
    return DTO_OK;
}

// Every interval kernel of the problem honours DProb::kc0/kc1 (the persistent and octet bilinear variants and the
// time-dependent kernels do).  Cross-knot Hessian blocks (time-dependent integrator, linear spline) are fine: the assembler
// of a range reads the compact second derivatives of interval kc0 - 1, which the range before it wrote.
static bool range_capable(const dto_handle* h) {
    const DProb& P = h->P;
    if (P.batch != 1 || P.gl.G > 0) return false;
    for (int i = 0; i < P.n_int; ++i) {
        const DInt& I = P.in[i];
        if (I.kind == DTO_INT_DERIVATIVE || I.kind == DTO_INT_TDBILINEAR) continue;
        if (!(I.kind == DTO_INT_BILINEAR && I.variant >= DTO_VAR_PERSISTENT)) return false;
    }
    return true;
}

extern "C" int dto_eval_all_dev(dto_handle* h, const double* dZ, double sigma, const double* dmu, double* dJ, double* dgrad,
                                double* dg, double* djac, double* dhess) {
    if (!h || !dZ) return DTO_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    // scratch shared with the cached callbacks (compact Hessian, jets) is overwritten; caller-owned outputs are not tracked
    if (dZ != h->dZ) h->have_jets = false;
    return run_eval(h, dZ, sigma, dmu, dJ, dgrad, dg, djac, dhess);
}

extern "C" int dto_synchronize(dto_handle* h) {
    if (!h) return DTO_ERR_INVALID;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return check_link_errors(h);
}

// ---- iterate cache -----------------------------------------------------------------------------------
// 1: Z is the resident iterate (nothing moved); 0: a new iterate was uploaded (every cached quantity dropped); < 0: error
static int publish_iterate(dto_handle* h, const double* src);
static int ensure_iterate(dto_handle* h, const double* Z, bool force = false) {
    const DProb& P = h->P;
    const size_t bytes = sizeof(double) * (size_t)P.batch * (size_t)P.n_vars_local;
    if (!force && h->z_valid && memcmp(h->hZpin, Z, bytes) == 0) {
        ++h->cache_hits;
        return 1;
    }
    ++h->cache_misses;
    if (h->async_inflight && !h->prefetch_consumed) h->prefetch_score = -4;  // an early start nobody used: pause them
    h->prefetch_consumed = false;
    h->g_staged = false;
    h->have_obj = h->have_g = h->have_jac = h->have_jets = false;
    h->z_valid = false;
    h->spec_jac_done = false;
    if (h->spec_jac_inflight) {  // the previous iterate's Jacobian is still leaving for the registered array
        CUDA_TRY(h, cudaStreamSynchronize(h->copy_stream));
        h->spec_jac_inflight = false;
    }
    memcpy(h->hZpin, Z, bytes);
    CUDA_TRY(h, cudaMemcpyAsync(h->dZ, h->hZpin, bytes, cudaMemcpyHostToDevice, h->stream));
    h->z_valid = true;
    const int rc = publish_iterate(h, h->dZ);
    return rc < 0 ? rc : 0;
}

extern "C" int dto_cache_stats(const dto_handle* h, int64_t* hits, int64_t* misses) {
    if (!h || !hits || !misses) return DTO_ERR_INVALID;
    *hits = h->cache_hits;
    *misses = h->cache_misses;
    return DTO_OK;
}

extern "C" int dto_upload(dto_handle* h, const double* Z) {
    if (!h || !Z) return DTO_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    // linked shards count iterates in lockstep: every dto_upload is a new iterate on every rank, changed or not
    const int rc = ensure_iterate(h, Z, h->link_rank >= 0);
    if (rc < 0) return rc;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DTO_OK;
}

extern "C" int dto_upload_dev(dto_handle* h, const double* dZ) {
    if (!h || !dZ) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    CUDA_TRY(h, cudaSetDevice(h->device));
    h->have_obj = h->have_g = h->have_jac = h->have_jets = h->g_staged = false;
    h->z_valid = false;  // the host copy no longer describes the resident iterate
    if (h->link_rank >= 0 && h->link_world > 1) return publish_iterate(h, dZ);  // copy + publish (+ wait) in one kernel
    if (dZ != h->dZ)
        CUDA_TRY(h, cudaMemcpyAsync(h->dZ, dZ, sizeof(double) * (size_t)P.batch * (size_t)P.n_vars_local, cudaMemcpyDeviceToDevice, h->stream));
    return publish_iterate(h, h->dZ);
}

// joins the zero-fill workers on every exit path (they write into the caller's buffer)
struct FillGuard {
    ZeroFill* z = nullptr;
    ~FillGuard() {
        if (z) z->finish();
    }
};

// DTO_B200_TRACE: timestamps (CUDA events) of the stages of one host-pointer call, printed relative to its first event
struct Tracer {
    bool on;
    std::vector<std::pair<const char*, cudaEvent_t>> ev;
    explicit Tracer(bool o) : on(o) {}
    void mark(const char* what, cudaStream_t st) {
        if (!on) return;
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        cudaEventRecord(e, st);
        ev.emplace_back(what, e);
    }
    ~Tracer() {
        if (!on || ev.empty()) return;
        cudaDeviceSynchronize();
        std::string line = "[dto trace]";
        for (size_t i = 1; i < ev.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[0].second, ev[i].second);
            char buf[96];
            snprintf(buf, sizeof(buf), " %s %.0fus", ev[i].first, ms * 1e3);
            line += buf;
        }
        fprintf(stderr, "%s\n", line.c_str());
        for (auto& e : ev) cudaEventDestroy(e.second);
    }
};

// What one host-pointer call computes on the device (`passes`, `comp_obj`) and what it delivers to the caller (the non-null
// host pointers).  Z (and mu) are already on their way to the device.  A quantity that is delivered but not computed is
// resident from an earlier callback on the same iterate.  `spec_jac`: the Jacobian computed by this call also goes to the
// registered array on the copy stream, and the call returns without waiting for it (dto_eval_jacobian on the same iterate
// with that array only joins the copy).
static int eval_core(dto_handle* h, double sigma, const EvalFlags* passes, int n_passes, bool comp_obj, double* J, double* grad,
                     double* g, double* jac, double* hess, bool spec_jac = false, bool prefetch = false) {
    h->g_ready_valid = false;
    {
        const int rc0 = prepare_halo(h);
        if (rc0 != DTO_OK) return rc0;
    }
    const DProb& P = h->P;
    const size_t B = (size_t)P.batch;
    bool comp_jac = false, comp_hess = false, comp_g = false;
    for (int i = 0; i < n_passes; ++i) {
        comp_g |= passes[i].want_g;
        comp_jac |= passes[i].want_jac;
        comp_hess |= passes[i].want_hess;
    }
    begin_hs_exchange(h, comp_hess);
    if (spec_jac) jac = h->reg_jac;
    long long d2h = 8LL * B * ((J ? 1 : 0) + (grad ? P.n_grad_local : 0) + (g ? P.n_cons_local : 0));
    double* dJ = comp_obj ? h->dJ : nullptr;
    double* dgrad = comp_obj ? h->dgrad : nullptr;
    EvalFlags fany{comp_g, comp_jac, comp_hess};

    // Structural constants stay off the bus: a registered array has them in place (written once by dto_register_outputs);
    // an unregistered Hessian buffer gets them from the handle's host threads while the GPU computes.
    const bool reg_h = hess && hess == h->reg_hess && h->reg_hess_sparse;
    const bool reg_j = jac && jac == h->reg_jac && h->reg_jac_sparse;
    const bool big = 8LL * ((jac ? P.nnz_jac_local : 0) + (hess ? P.nnz_hess_local : 0)) >= (8LL << 20) && P.nI >= 512;
    const bool sparse_hess = hess && big && !h->hess_runs.empty() && (reg_h || (h->zero_fill && range_capable(h)));
    const bool sparse_jac = jac && big && reg_j && h->jac_skip_ok > 0;
    const bool fill_h = sparse_hess && !reg_h;

    // Jacobian columns / Hessian regions of the local knots [ka, kb) on stream `st`
    auto deliver_jac = [&](int ka, int kb, cudaStream_t st) -> int {
        auto whole = [&](int a, int b2) -> int {
            if (a >= b2) return DTO_OK;
            // the columns of the global variables follow the last knot's (evaluator.jl:123)
            const long long p0 = h->jac_colptr[(size_t)a * P.z], p1 = b2 >= P.nK ? P.nnz_jac_local : h->jac_colptr[(size_t)b2 * P.z];
            CUDA_TRY(h, cudaMemcpyAsync(jac + p0, h->djac + p0, sizeof(double) * (p1 - p0), cudaMemcpyDeviceToHost, st));
            d2h += 8LL * (p1 - p0);
            return DTO_OK;
        };
        if (!sparse_jac) return whole(ka, kb);
        // knot 0 and the last knot whole; inner knots: every column minus its constant head, one strided copy
        int rc = whole(ka, std::min(kb, 1));
        if (rc != DTO_OK) return rc;
        const int a = std::max(ka, 1), b2 = std::min(kb, P.nI);
        if (a < b2) {
            const long long Lc = 2LL * P.Dsum, sk = h->jac_skip_ok;
            const long long p0 = h->jac_colptr[(size_t)a * P.z] + sk;
            CUDA_TRY(h, cudaMemcpy2DAsync(jac + p0, sizeof(double) * Lc, h->djac + p0, sizeof(double) * Lc, sizeof(double) * (Lc - sk),
                                          (size_t)(b2 - a) * P.z, cudaMemcpyDeviceToHost, st));
            d2h += 8LL * (Lc - sk) * (b2 - a) * P.z;
        }
        return whole(std::max(ka, P.nI), kb);
    };
    auto deliver_hess = [&](int ka, int kb, cudaStream_t st) -> int {
        kb = std::min(kb, P.nOwn);
        if (ka >= kb) return DTO_OK;
        if (!sparse_hess) {
            const long long p0 = hess_knot_base(P, ka), p1 = kb >= P.nOwn ? P.nnz_hess_local : hess_knot_base(P, kb);
            CUDA_TRY(h, cudaMemcpyAsync(hess + p0, h->dhess + p0, sizeof(double) * (p1 - p0), cudaMemcpyDeviceToHost, st));
            d2h += 8LL * (p1 - p0);
            return DTO_OK;
        }
        // only the columns >= l0 of every knot of the range: one 2-D copy per run of equal knots
        for (const HRun& r : h->hess_runs) {
            const int a = std::max(r.k0, ka), b2 = std::min(r.k0 + r.cnt, kb);
            if (a >= b2) continue;
            const long long nc = hess_knot_has_cross(P, a) ? P.z : 0;
            const long long region = nc * P.z + (long long)P.z * (P.z + 1) / 2;
            const long long skip = (long long)r.l0 * nc + (long long)r.l0 * (r.l0 + 1) / 2;
            if (region == skip) continue;
            const long long p0 = hess_knot_base(P, a) + skip;
            CUDA_TRY(h, cudaMemcpy2DAsync(hess + p0, sizeof(double) * region, h->dhess + p0, sizeof(double) * region,
                                          sizeof(double) * (region - skip), (size_t)(b2 - a), cudaMemcpyDeviceToHost, st));
            d2h += 8LL * (region - skip) * (b2 - a);
        }
        return DTO_OK;
    };

    // early start: the residual goes to a page-locked staging buffer as soon as it is complete -- issued BEFORE the last
    // block of the speculative Jacobian delivery, or the constraint callback would queue behind it on the copy engine
    auto stage_g = [&]() -> int {
        if (!prefetch || !comp_g || B != 1) return DTO_OK;
        if (!h->hg_pin && cudaHostAlloc((void**)&h->hg_pin, sizeof(double) * (size_t)std::max<long long>(1, P.n_cons_local), cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            h->hg_pin = nullptr;
            return DTO_OK;  // no staging: the constraint callback copies from the device
        }
        CUDA_TRY(h, cudaMemcpyAsync(h->hg_pin, h->dg, sizeof(double) * P.n_cons_local, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaEventRecord(h->ev_g, h->stream));
        d2h += 8LL * P.n_cons_local;
        h->g_staged = true;
        return DTO_OK;
    };

    Tracer tr(h->trace != 0);
    tr.mark("start", h->stream);
    // series plans of this iterate (a Hessian pass from stored jets re-uses the plans of the pass that stored them)
    if ((comp_g || comp_jac || comp_hess) && !(n_passes == 1 && passes[0].jets == DTO_JETS_USE)) launch_plans(h, P, h->dZ);
    FillGuard guard;
    if (fill_h) {
        // host threads write the structural zeros into the caller's Hessian buffer while the GPU computes
        const dto_handle* hh = h;
        double* hz = hess;
        h->zero_fill->launch([hh, hz](int part, int parts) {
            const size_t n = hh->hess_zero_segs.size(), lo = n * part / parts, hi = n * (part + 1) / parts;
            for (size_t i = lo; i < hi; ++i)
                memset(hz + hh->hess_zero_segs[i].first, 0, sizeof(double) * (size_t)hh->hess_zero_segs[i].second);
        });
        guard.z = h->zero_fill;  // joined on every exit path below
    }

    // Large sparse outputs that are computed by this call: cut the trajectory into a few knot ranges; the Jacobian columns
    // and Hessian blocks of a finished range go out on the copy engine while the next range is being computed.
    // (`jac` includes the registered array of a speculative delivery)
    const long long out_bytes = 8LL * ((jac && comp_jac ? P.nnz_jac_local : 0) + (hess && comp_hess ? P.nnz_hess_local : 0));
    const bool pipelined = !h->pipeline_fracs.empty() && out_bytes >= (8LL << 20) && P.nI >= 512 && range_capable(h) &&
                           !(n_passes == 1 && passes[0].jets == DTO_JETS_USE);  // the adjoint-only pass is too short to be worth cutting
    bool used_copy_stream = false;
    int rc = DTO_OK;
    // a resident Jacobian asked for (not computed here): right away, beside the computation
    if (jac && !comp_jac) {
        if (B == 1) {
            used_copy_stream = true;
            if ((rc = deliver_jac(0, P.nK, h->copy_stream)) != DTO_OK) return rc;
        } else {
            CUDA_TRY(h, cudaMemcpyAsync(jac, h->djac, sizeof(double) * B * P.nnz_jac_local, cudaMemcpyDeviceToHost, h->stream));
            d2h += 8LL * B * P.nnz_jac_local;
        }
    }
    if (prefetch) {
        // early start: the objective and its gradient first, on their way to the host before the interval kernels begin
        eval_prologue(h, P, h->dZ, dJ, dgrad, nullptr, nullptr, EvalFlags{false, false, false});
        if (J) CUDA_TRY(h, cudaMemcpyAsync(J, h->dJ, sizeof(double) * B, cudaMemcpyDeviceToHost, h->stream));
        if (grad) CUDA_TRY(h, cudaMemcpyAsync(grad, h->dgrad, sizeof(double) * B * P.n_grad_local, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaEventRecord(h->ev_small, h->stream));
        J = grad = nullptr;
        dJ = dgrad = nullptr;
    }
    if (!pipelined) {
        for (int i = 0; i < n_passes; ++i)
            if ((rc = eval_range(h, P, h->dZ, sigma, h->dmu, h->dg, h->djac, h->dhess, passes[i])) != DTO_OK) return rc;
        eval_prologue(h, P, h->dZ, dJ, dgrad, h->dg, h->djac, fany);
        CUDA_TRY(h, cudaGetLastError());
        if ((rc = stage_g()) != DTO_OK) return rc;
        if (B == 1) {
            cudaStream_t jst = h->stream;
            if (spec_jac && comp_jac) {  // the speculative copy must not hold up this call's own outputs
                CUDA_TRY(h, cudaEventRecord(h->chunk_events_at(0), h->stream));
                CUDA_TRY(h, cudaStreamWaitEvent(h->copy_stream, h->chunk_events_at(0), 0));
                jst = h->copy_stream;
                used_copy_stream = true;
            }
            if (jac && comp_jac && (rc = deliver_jac(0, P.nK, jst)) != DTO_OK) return rc;
            if (hess && (rc = deliver_hess(0, P.nOwn, h->stream)) != DTO_OK) return rc;
        } else {
            if (jac && comp_jac) CUDA_TRY(h, cudaMemcpyAsync(jac, h->djac, sizeof(double) * B * P.nnz_jac_local, cudaMemcpyDeviceToHost, h->stream));
            if (hess) CUDA_TRY(h, cudaMemcpyAsync(hess, h->dhess, sizeof(double) * B * P.nnz_hess_local, cudaMemcpyDeviceToHost, h->stream));
            if (hess) d2h += 8LL * B * P.nnz_hess_local;
            if (jac && comp_jac) d2h += 8LL * B * P.nnz_jac_local;
        }
    } else {
        used_copy_stream = true;
        std::vector<int> bounds{0};
        for (double fr : h->pipeline_fracs) {
            const int k = (int)(fr * P.nI);
            if (k > bounds.back() && k < P.nI) bounds.push_back(k);
        }
        bounds.push_back(P.nK);
        const bool jac_now = jac && comp_jac, hess_now = hess && comp_hess;
        eval_prologue(h, P, h->dZ, dJ, dgrad, h->dg, h->djac, fany);  // knot-constraint entries land before any column leaves
        DProb Pr = P;
        for (size_t c = 0; c + 1 < bounds.size(); ++c) {
            Pr.kc0 = bounds[c];
            Pr.kc1 = bounds[c + 1];
            for (int i = 0; i < n_passes; ++i)
                if ((rc = eval_range(h, Pr, h->dZ, sigma, h->dmu, h->dg, h->djac, h->dhess, passes[i])) != DTO_OK) return rc;
            cudaEvent_t ev = h->chunk_events_at(c);
            if (!ev) {
                h->err = "cudaEventCreate failed";
                return DTO_ERR_CUDA;
            }
            CUDA_TRY(h, cudaEventRecord(ev, h->stream));
            tr.mark("range-computed", h->stream);
            if (spec_jac && c + 2 == bounds.size()) {
                // last range of a speculative delivery: the outputs this call was asked for (a few hundred KB) go to the copy
                // engine BEFORE the last block of the Jacobian nobody is waiting for yet
                if (J) CUDA_TRY(h, cudaMemcpyAsync(J, h->dJ, sizeof(double) * B, cudaMemcpyDeviceToHost, h->stream));
                if (grad) CUDA_TRY(h, cudaMemcpyAsync(grad, h->dgrad, sizeof(double) * B * P.n_grad_local, cudaMemcpyDeviceToHost, h->stream));
                if (g) CUDA_TRY(h, cudaMemcpyAsync(g, h->dg, sizeof(double) * B * P.n_cons_local, cudaMemcpyDeviceToHost, h->stream));
                J = grad = g = nullptr;
                if ((rc = stage_g()) != DTO_OK) return rc;
                cudaEvent_t ev2 = h->chunk_events_at(bounds.size());
                if (!ev2) {
                    h->err = "cudaEventCreate failed";
                    return DTO_ERR_CUDA;
                }
                CUDA_TRY(h, cudaEventRecord(ev2, h->stream));
                ev = ev2;
            }
            CUDA_TRY(h, cudaStreamWaitEvent(h->copy_stream, ev, 0));
            // columns of knots [kc0, kc1): their own-interval rows were written by this range, the previous-interval rows
            // of knot kc0 by the range before
            if (jac_now && (rc = deliver_jac(Pr.kc0, Pr.kc1, h->copy_stream)) != DTO_OK) return rc;
            if (hess_now && h->hs_recv_now) {  // the first knot is assembled after the last range (eval_range): it leaves last
                if ((rc = deliver_hess(std::max(Pr.kc0, 1), Pr.kc1, h->copy_stream)) != DTO_OK) return rc;
                if (Pr.kc1 >= P.nK && (rc = deliver_hess(0, 1, h->copy_stream)) != DTO_OK) return rc;
            } else if (hess_now && (rc = deliver_hess(Pr.kc0, Pr.kc1, h->copy_stream)) != DTO_OK) {
                return rc;
            }
            tr.mark("range-delivered", h->copy_stream);
        }
        CUDA_TRY(h, cudaGetLastError());
    }
    if (J) CUDA_TRY(h, cudaMemcpyAsync(J, h->dJ, sizeof(double) * B, cudaMemcpyDeviceToHost, h->stream));
    if (grad) CUDA_TRY(h, cudaMemcpyAsync(grad, h->dgrad, sizeof(double) * B * P.n_grad_local, cudaMemcpyDeviceToHost, h->stream));
    if (g) CUDA_TRY(h, cudaMemcpyAsync(g, h->dg, sizeof(double) * B * P.n_cons_local, cudaMemcpyDeviceToHost, h->stream));
    tr.mark("main-stream-done", h->stream);
    // everything is enqueued: the calling thread writes its share of the structural zeros while the GPU works
    if (guard.z) {
        guard.z->finish();
        guard.z = nullptr;
    }
    if (prefetch) {  // only this call's own small outputs are waited for; the pass runs on
        CUDA_TRY(h, cudaEventSynchronize(h->ev_small));
        if (spec_jac) h->spec_jac_inflight = true;
        h->async_inflight = true;
        h->last_d2h_bytes = d2h;
        return DTO_OK;
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->async_inflight = false;
    if (spec_jac) h->spec_jac_inflight = true;
    else if (used_copy_stream) {  // (an earlier call's speculative Jacobian copy stays in flight: the Jacobian callback waits for it)
        CUDA_TRY(h, cudaStreamSynchronize(h->copy_stream));
        h->spec_jac_inflight = false;
    }
    h->last_d2h_bytes = d2h;
    return check_link_errors(h);
}

// One fused pass over one iterate (benchmark/benchmarks.jl:23-38 times the five callbacks on one iterate; a solver calls
// them separately: see the single callbacks below).
extern "C" int dto_eval_all(dto_handle* h, const double* Z, double sigma, const double* mu, double* J, double* grad, double* g,
                            double* jac, double* hess) {
    if (!h || !Z) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    int rc = check_eval_args(h, mu, hess);
    if (rc != DTO_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if ((rc = ensure_iterate(h, Z)) < 0) return rc;
    // the fused pass recomputes what it is asked for and leaves the callbacks' cache empty (its Hessian pass overwrites
    // the compact second derivatives with this call's mu)
    h->have_obj = h->have_g = h->have_jac = h->have_jets = h->g_staged = false;
    if (hess) CUDA_TRY(h, cudaMemcpyAsync(h->dmu, mu, sizeof(double) * (size_t)P.batch * P.n_cons_local, cudaMemcpyHostToDevice, h->stream));
    EvalFlags f{g != nullptr, jac != nullptr, hess != nullptr};
    rc = eval_core(h, sigma, &f, 1, J || grad, J, grad, g, jac, hess);
    if (rc == DTO_OK) {
        h->have_obj = J || grad;
        h->have_g = g;
        h->have_jac = jac;
    }
    return rc;
}

// The five callbacks as a solver calls them: separately, usually on one iterate (f, grad f, g, jac g, then the Hessian
// with the new multipliers).  The first callback that needs the interval kernels on a NEW iterate runs ONE mu-independent
// pass (residual + Jacobian; the forward role also stores the second-order vectors of its jet); later callbacks on the
// same iterate only copy, and the Hessian callback runs the adjoint role, contracts the stored jets with mu and assembles.
static int eval_callback(dto_handle* h, const double* Z, double sigma, const double* mu, double* J, double* grad, double* g,
                         double* jac, double* hess) {
    if (!h || !Z) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    int rc = check_eval_args(h, mu, hess);
    if (rc != DTO_OK) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if ((rc = ensure_iterate(h, Z)) < 0) return rc;
    if (jac && jac == h->reg_jac && h->have_jac && h->spec_jac_done && !J && !grad && !g && !hess) {
        // the Jacobian of this iterate went to the registered array while the constraint callback computed it
        h->prefetch_consumed = true;
        if (h->spec_jac_inflight) {
            CUDA_TRY(h, cudaStreamSynchronize(h->copy_stream));
            h->spec_jac_inflight = false;
        }
        h->last_d2h_bytes = 0;
        return DTO_OK;
    }
    const bool only_small = (J || grad) && !g && !jac && !hess;
    if (only_small && h->have_obj && h->async_inflight) {
        // resident objective / gradient while an early-started pass still runs on the main stream: a side stream ordered
        // after the objective kernels only
        CUDA_TRY(h, cudaStreamWaitEvent(h->aux_stream, h->ev_small, 0));
        if (J) CUDA_TRY(h, cudaMemcpyAsync(J, h->dJ, sizeof(double) * P.batch, cudaMemcpyDeviceToHost, h->aux_stream));
        if (grad) CUDA_TRY(h, cudaMemcpyAsync(grad, h->dgrad, sizeof(double) * (size_t)P.batch * P.n_grad_local, cudaMemcpyDeviceToHost, h->aux_stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->aux_stream));
        h->last_d2h_bytes = 8LL * P.batch * ((J ? 1 : 0) + (grad ? P.n_grad_local : 0));
        return DTO_OK;
    }
    if (g && !J && !grad && !jac && !hess && h->have_g && h->g_staged) {
        // the residual of this iterate was staged by the early-started pass
        h->prefetch_consumed = true;
        if (h->prefetch_score < 0) h->prefetch_score = 0;
        CUDA_TRY(h, cudaEventSynchronize(h->ev_g));
        memcpy(g, h->hg_pin, sizeof(double) * (size_t)P.n_cons_local);
        h->last_d2h_bytes = 0;  // counted by the call that staged it
        return DTO_OK;
    }
    if ((g || jac || hess) && h->async_inflight && (h->have_g || h->have_jac)) {
        h->prefetch_consumed = true;
        if (h->prefetch_score < 0) h->prefetch_score = 0;
    } else if ((g || jac) && !h->have_g && !h->have_jac && h->have_obj && h->prefetch_score < 0) {
        ++h->prefetch_score;  // the objective came first on this iterate and the pass was needed after all: an early start would have paid
    }
    EvalFlags passes[2];
    int np = 0;
    const bool comp_obj = (J || grad) && !h->have_obj;
    // early start: the first callback on a new iterate asks for the objective or its gradient only
    const bool prefetch = only_small && comp_obj && !h->have_g && !h->have_jac && P.batch == 1 && h->link_rank < 0 &&
                          h->prefetch_score >= 0 && P.nI >= 256 && h->jets_ok;
    const bool use_jets = hess && h->jets_ok;
    const bool need_g = g && !h->have_g, need_jac = jac && !h->have_jac;
    const bool need_jets = use_jets && !h->have_jets;
    if (need_g || need_jac || need_jets || prefetch) {
        // the one mu-independent pass of this iterate: residual + Jacobian (+ the jets the Hessian callback uses)
        EvalFlags f1{true, true, false};
        f1.jets = h->jets_ok ? DTO_JETS_STORE : DTO_JETS_NONE;
        passes[np++] = f1;
    }
    if (hess) {
        CUDA_TRY(h, cudaMemcpyAsync(h->dmu, mu, sizeof(double) * (size_t)P.batch * P.n_cons_local, cudaMemcpyHostToDevice, h->stream));
        EvalFlags f2{false, false, true};
        f2.jets = use_jets ? DTO_JETS_USE : DTO_JETS_NONE;
        passes[np++] = f2;
    }
    // a Jacobian that is computed without being asked for goes to the registered array on the side
    const bool spec = !jac && h->reg_jac != nullptr && np > 0 && passes[0].want_jac && P.batch == 1;
    rc = eval_core(h, sigma, passes, np, comp_obj, J, grad, g, jac, hess, spec, prefetch);
    if (rc != DTO_OK) {
        h->have_obj = h->have_g = h->have_jac = h->have_jets = h->g_staged = false;
        h->async_inflight = false;
        return rc;
    }
    if (spec) h->spec_jac_done = true;
    if (jac && jac == h->reg_jac) h->spec_jac_done = true;
    if (comp_obj) h->have_obj = true;
    for (int i = 0; i < np; ++i) {
        h->have_g |= passes[i].want_g;
        h->have_jac |= passes[i].want_jac;
        h->have_jets |= passes[i].jets == DTO_JETS_STORE;
    }
    return DTO_OK;
}

extern "C" int dto_eval_objective(dto_handle* h, const double* Z, double* J) {
    if (!J) return DTO_ERR_INVALID;
    return eval_callback(h, Z, 0.0, nullptr, J, nullptr, nullptr, nullptr, nullptr);
}
extern "C" int dto_eval_gradient(dto_handle* h, const double* Z, double* grad) {
    if (!grad) return DTO_ERR_INVALID;
    return eval_callback(h, Z, 0.0, nullptr, nullptr, grad, nullptr, nullptr, nullptr);
}
extern "C" int dto_eval_constraint(dto_handle* h, const double* Z, double* g) {
    if (!g) return DTO_ERR_INVALID;
    return eval_callback(h, Z, 0.0, nullptr, nullptr, nullptr, g, nullptr, nullptr);
}
extern "C" int dto_eval_jacobian(dto_handle* h, const double* Z, double* vals) {
    if (!vals) return DTO_ERR_INVALID;
    return eval_callback(h, Z, 0.0, nullptr, nullptr, nullptr, nullptr, vals, nullptr);
}
extern "C" int dto_eval_hessian(dto_handle* h, const double* Z, double sigma, const double* mu, double* vals) {
    if (!vals) return DTO_ERR_INVALID;
    return eval_callback(h, Z, sigma, mu, nullptr, nullptr, nullptr, nullptr, vals);
}

// ---- registered outputs ------------------------------------------------------------------------------
static void unpin(bool& pinned, double*& p) {
    if (pinned && p) {
        cudaHostUnregister(p);
        cudaGetLastError();
    }
    pinned = false;
    p = nullptr;
}

extern "C" int dto_unregister_outputs(dto_handle* h) {
    if (!h) return DTO_ERR_INVALID;
    cudaSetDevice(h->device);
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    h->spec_jac_inflight = h->spec_jac_done = false;
    unpin(h->reg_jac_pinned, h->reg_jac);
    unpin(h->reg_hess_pinned, h->reg_hess);
    h->reg_jac_sparse = h->reg_hess_sparse = false;
    return DTO_OK;
}

extern "C" int dto_register_outputs(dto_handle* h, double* jac_vals, double* hess_vals) {
    if (!h) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    CUDA_TRY(h, cudaSetDevice(h->device));
    dto_unregister_outputs(h);
    if (P.batch != 1) {
        h->err = "dto_register_outputs: one problem per handle (batch == 1)";
        return DTO_ERR_UNSUPPORTED;
    }
    auto pin = [&](double* p, long long n, bool& pinned) {
        const cudaError_t e = cudaHostRegister(p, sizeof(double) * (size_t)n, cudaHostRegisterPortable);
        pinned = e == cudaSuccess;
        cudaGetLastError();  // already page-locked by the caller (or not lockable): the copies still work
    };
    if (jac_vals) {
        pin(jac_vals, P.nnz_jac_local, h->reg_jac_pinned);
        h->reg_jac = jac_vals;
        if (h->jac_skip_ok > 0) {
            // head of every column of the inner knots: the previous-interval block of the first integrator, [0 .. 1 .. 0]
            const int d1 = h->jac_skip_ok, xo = P.in[0].x_off;
            for (long long kl = 1; kl < P.nI; ++kl)
                for (int l = 0; l < P.z; ++l) {
                    double* c = jac_vals + h->jac_colptr[(size_t)kl * P.z + l];
                    memset(c, 0, sizeof(double) * (size_t)d1);
                    if (l >= xo && l < xo + d1) c[l - xo] = 1.0;
                }
            h->reg_jac_sparse = true;
        }
    }
    if (hess_vals && h->eval_hessian) {
        pin(hess_vals, P.nnz_hess_local, h->reg_hess_pinned);
        h->reg_hess = hess_vals;
        if (!h->hess_runs.empty()) {
            for (const auto& sgm : h->hess_zero_segs) memset(hess_vals + sgm.first, 0, sizeof(double) * (size_t)sgm.second);
            h->reg_hess_sparse = true;
        }
    }
    return DTO_OK;
}

// Products straight from the series for problems made of persistent-variant bilinear integrators, derivative
// integrators and knot constraints; anything else materialises the Jacobian values first, as the reference does
// (evaluator.jl:406-456).  DTO_B200_JVP=materialize forces the latter.
static bool matrix_free_capable(const dto_handle* h) {
    const DProb& P = h->P;
    if (h->sharded || P.gl.G > 0) return false;
    const char* env = getenv("DTO_B200_JVP");
    if (env && strcmp(env, "materialize") == 0) return false;
    for (int i = 0; i < P.n_int; ++i)
        if (P.in[i].kind != DTO_INT_DERIVATIVE && !(P.in[i].kind == DTO_INT_BILINEAR && P.in[i].variant >= DTO_VAR_PERSISTENT)) return false;
    return true;
}

static int jac_product(dto_handle* h, const double* Z, const double* w, double* y, bool transpose) {
    if (!h || !Z || !w || !y) return DTO_ERR_INVALID;
    const DProb& P = h->P;
    const size_t B = (size_t)P.batch;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->sharded) {
        h->err = "Jacobian products are not available on knot-range shards";
        return DTO_ERR_UNSUPPORTED;
    }
    if (!h->dw) {
        h->dw = dev_upload<double>(h, nullptr, B * (size_t)std::max(P.n_vars_local, P.n_cons_local));
        h->dy = dev_upload<double>(h, nullptr, B * (size_t)std::max(P.n_vars_local, P.n_cons_local));
        if (!h->dw || !h->dy) {
            h->err = "device allocation failed (Jacobian product)";
            return DTO_ERR_ALLOC;
        }
    }
    const size_t nw = transpose ? (size_t)P.n_cons_local : (size_t)P.n_vars_local;
    const size_t ny = transpose ? (size_t)P.n_vars_local : (size_t)P.n_cons_local;
    {
        const int rc = ensure_iterate(h, Z);
        if (rc < 0) return rc;
    }
    CUDA_TRY(h, cudaMemcpyAsync(h->dw, w, sizeof(double) * B * nw, cudaMemcpyHostToDevice, h->stream));
    bool done = false;
    if (matrix_free_capable(h)) {
        CUDA_TRY(h, cudaMemsetAsync(h->dy, 0, sizeof(double) * B * ny, h->stream));
        done = true;
        for (int i = 0; i < P.n_int && done; ++i)
            if (P.in[i].kind == DTO_INT_BILINEAR) done = launch_bilinear_product(P, i, h->dZ, h->dw, h->dy, transpose, h->stream, &h->launches);
        if (done) launch_analytic_product(P, h->dZ, h->dw, h->dy, transpose, h->stream, &h->launches);
    }
    if (!done) {
        if (!h->d_rows0) {
            std::vector<int64_t> r((size_t)P.nnz_jac_local), c((size_t)P.nnz_jac_local);
            int rc = dto_jac_structure(h, r.data(), c.data());
            if (rc != DTO_OK) return rc;
            for (auto& v : r) v -= 1;  // a whole-problem handle has local == global numbering
            for (auto& v : c) v -= 1;
            h->d_rows0 = (long long*)dev_upload(h, (const long long*)r.data(), r.size());
            h->d_cols0 = (long long*)dev_upload(h, (const long long*)c.data(), c.size());
            if (!h->d_rows0 || !h->d_cols0) {
                h->err = "device allocation failed (Jacobian product)";
                return DTO_ERR_ALLOC;
            }
        }
        if (!h->have_jac) {
            int rc = run_eval(h, h->dZ, 0.0, nullptr, nullptr, nullptr, nullptr, h->djac, nullptr);
            if (rc != DTO_OK) return rc;
            h->have_jac = true;
        }
        launch_jac_product(P, h->djac, h->d_rows0, h->d_cols0, h->dw, h->dy, transpose, h->stream, &h->launches);
    }
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemcpyAsync(y, h->dy, sizeof(double) * B * ny, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DTO_OK;
}
extern "C" int dto_eval_jacobian_product(dto_handle* h, const double* Z, const double* w, double* y) {
    return jac_product(h, Z, w, y, false);
}
extern "C" int dto_eval_jacobian_transpose_product(dto_handle* h, const double* Z, const double* w, double* y) {
    return jac_product(h, Z, w, y, true);
}

extern "C" int dto_violation_dev(dto_handle* h, const double* dg, double* dviol) {
    if (!h || !dg || !dviol) return DTO_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    launch_violation(h->P, dg, h->d_row_is_eq, dviol, h->stream, &h->launches);
    CUDA_TRY(h, cudaGetLastError());
    return DTO_OK;
}

// ---- links between knot-range shards ---------------------------------------------------------------------
extern "C" double* dto_local_Z(dto_handle* h) { return h ? h->dZ : nullptr; }

// the halo slots [2][z], then the boundary Hessian block slots [2][hblk_len]: the same size on every shard of a problem
static size_t xwin_bytes(const dto_handle* h) { return sizeof(XWin) + sizeof(double) * 2 * ((size_t)h->P.z + (size_t)h->hblk_len); }

static int ensure_xwin(dto_handle* h) {
    if (h->xwin) return DTO_OK;
    void* p = nullptr;
    CUDA_TRY(h, cudaMalloc(&p, xwin_bytes(h)));  // its own allocation: the IPC handle exposes nothing else
    h->allocs.push_back(p);
    CUDA_TRY(h, cudaMemset(p, 0, xwin_bytes(h)));
    h->xwin = (XWin*)p;
    return DTO_OK;
}

extern "C" int dto_shard_export(dto_handle* h, void* out64) {
    if (!h || !out64) return DTO_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    int rc = ensure_xwin(h);
    if (rc != DTO_OK) return rc;
    cudaIpcMemHandle_t mh;
    CUDA_TRY(h, cudaIpcGetMemHandle(&mh, h->xwin));
    static_assert(sizeof(mh) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(out64, &mh, 64);
    return DTO_OK;
}

static int finish_link(dto_handle* h, int rank, int world) {
    h->link_rank = rank;
    h->link_world = world;
    h->epoch = h->waited_epoch = h->scal_seq = h->hseq = 0;
    h->z_valid = false;  // the next callback uploads (and publishes) whatever it is given
    if (!h->d_peer_win) {
        void* p = nullptr;
        CUDA_TRY(h, cudaMalloc(&p, sizeof(XWin*) * DTO_MAX_RANKS));
        h->allocs.push_back(p);
        h->d_peer_win = (XWin**)p;
    }
    CUDA_TRY(h, cudaMemcpy(h->d_peer_win, h->peer_win, sizeof(XWin*) * DTO_MAX_RANKS, cudaMemcpyHostToDevice));
    return DTO_OK;
}

static void drop_links(dto_handle* h) {
    for (int r = 0; r < DTO_MAX_RANKS; ++r) {
        if (h->peer_ipc[r] && h->peer_win[r]) cudaIpcCloseMemHandle(h->peer_win[r]);
        h->peer_ipc[r] = false;
        h->peer_win[r] = nullptr;
    }
    cudaGetLastError();
    h->link_rank = -1;
    h->link_world = 0;
    h->link_ipc = false;
    h->P.halo = nullptr;
}

extern "C" int dto_shard_link(dto_handle* h, int rank, int world, const void* handles64) {
    if (!h || !handles64 || world < 1 || world > DTO_MAX_RANKS || rank < 0 || rank >= world) return DTO_ERR_INVALID;
    if (!h->sharded) {
        h->err = "dto_shard_link: the handle is not a knot-range shard";
        return DTO_ERR_INVALID;
    }
    CUDA_TRY(h, cudaSetDevice(h->device));
    int rc = ensure_xwin(h);
    if (rc != DTO_OK) return rc;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    drop_links(h);  // a second link closes the first mappings
    // a re-link starts from a clean window: tags left by the previous link would let the first waits pass on stale data
    // (callers synchronise all ranks after linking, before anyone publishes into this window)
    CUDA_TRY(h, cudaMemset(h->xwin, 0, xwin_bytes(h)));
    for (int r = 0; r < world; ++r) {
        if (r == rank) {
            h->peer_win[r] = h->xwin;
            continue;
        }
        cudaIpcMemHandle_t mh;
        memcpy(&mh, (const char*)handles64 + 64 * (size_t)r, 64);
        void* p = nullptr;
        CUDA_TRY(h, cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess));
        h->peer_win[r] = (XWin*)p;
        h->peer_ipc[r] = true;
    }
    h->link_ipc = world > 1;
    return finish_link(h, rank, world);
}

extern "C" int dto_shard_link_local(dto_handle* const* hs, int world) {
    if (!hs || world < 1 || world > DTO_MAX_RANKS) return DTO_ERR_INVALID;
    for (int r = 0; r < world; ++r) {
        if (!hs[r] || !hs[r]->sharded) return DTO_ERR_INVALID;
        cudaSetDevice(hs[r]->device);
        int rc = ensure_xwin(hs[r]);
        if (rc != DTO_OK) return rc;
        cudaStreamSynchronize(hs[r]->stream);
        drop_links(hs[r]);
        CUDA_TRY(hs[r], cudaMemset(hs[r]->xwin, 0, xwin_bytes(hs[r])));  // a re-link starts from a clean window
    }
    for (int r = 0; r < world; ++r) {
        dto_handle* h = hs[r];
        CUDA_TRY(h, cudaSetDevice(h->device));
        for (int p = 0; p < world; ++p) {
            h->peer_win[p] = hs[p]->xwin;
            if (hs[p]->device != h->device) {
                cudaError_t e = cudaDeviceEnablePeerAccess(hs[p]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                    h->err = std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e);
                    return DTO_ERR_CUDA;
                }
                cudaGetLastError();
            }
        }
        int rc = finish_link(h, r, world);
        if (rc != DTO_OK) return rc;
    }
    return DTO_OK;
}

// A new iterate is on its way into dZ (stream order; src != dZ: the publish kernel copies it there): acknowledge the right
// neighbour's previous knot, push this shard's first knot to the left neighbour and -- shards linked across processes -- wait
// for the right neighbour's knot in the same kernel (every rank has its own host thread, so the spinning kernel cannot keep
// the neighbour from launching its push; shards linked inside one process wait in prepare_halo instead).
static int publish_iterate(dto_handle* h, const double* src) {
    if (h->link_rank < 0) return DTO_OK;
    ++h->epoch;
    XWin* left = h->link_rank > 0 ? h->peer_win[h->link_rank - 1] : nullptr;
    XWin* right = h->link_rank + 1 < h->link_world ? h->peer_win[h->link_rank + 1] : nullptr;
    const long long n = (long long)h->P.batch * h->P.n_vars_local;
    if (left || right || src != h->dZ) {
        launch_shard_publish(h->xwin, left, right, h->dZ, src, n, h->P.z, h->epoch, h->link_ipc, h->stream, &h->launches);
        if (h->link_ipc) h->waited_epoch = h->epoch;
    }
    CUDA_TRY(h, cudaGetLastError());
    return DTO_OK;
}

// Before the first kernel of an iterate that reads the halo knot: wait (on the device) until the right neighbour's push
// of this iterate has landed in this shard's window, and point the kernels at that slot.
static int prepare_halo(dto_handle* h) {
    if (h->link_rank < 0 || h->link_rank + 1 >= h->link_world) return DTO_OK;
    if (h->epoch == 0) {
        h->err = "linked shard: upload an iterate first (dto_upload / dto_upload_dev / any host-pointer callback)";
        return DTO_ERR_INVALID;
    }
    if (h->waited_epoch != h->epoch) {
        launch_shard_wait(h->xwin, h->epoch, h->stream, &h->launches);
        h->waited_epoch = h->epoch;
    }
    h->P.halo = h->xwin->halo + (size_t)(h->epoch & 1) * h->P.z;  // address arithmetic on a device pointer (no dereference)
    return DTO_OK;
}

static int check_link_errors(dto_handle* h) {
    if (h->link_rank < 0) return DTO_OK;
    unsigned long long e = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&e, &h->xwin->err, sizeof(e), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (e != 0) {
        switch (e) {
            case 1: h->err = "shard link: the left neighbour never released the halo slot (timeout)"; break;
            case 2: h->err = "shard link: the right neighbour's knot of this iterate never arrived (timeout); every rank must upload every iterate"; break;
            case 3: h->err = "shard link: scalar exchange timed out"; break;
            case 4:
                h->err = "shard link: Hessian exchange: the right neighbour never took the previous boundary block (timeout); a linked shard's "
                         "Hessian evaluation s reads what its left neighbour's evaluation s produced, so every rank evaluates every Hessian";
                break;
            default:
                h->err = "shard link: Hessian exchange: the left neighbour's boundary block of this Hessian evaluation never arrived (timeout); "
                         "a linked shard's Hessian evaluation s reads what its left neighbour's evaluation s produced, so every rank evaluates "
                         "every Hessian, and a thread that drives several linked shards calls them in rank order";
        }
        cudaMemsetAsync(&h->xwin->err, 0, sizeof(e), h->stream);
        return DTO_ERR_CUDA;
    }
    return DTO_OK;
}

extern "C" int dto_allreduce_scalars_dev(dto_handle* h, double* dJ, double* dviol) {
    if (!h || !dJ || !dviol) return DTO_ERR_INVALID;
    if (h->link_rank < 0) {
        h->err = "dto_allreduce_scalars_dev: the shard is not linked";
        return DTO_ERR_INVALID;
    }
    CUDA_TRY(h, cudaSetDevice(h->device));
    ++h->scal_seq;
    launch_scalar_exchange(h->xwin, h->d_peer_win, h->link_rank, h->link_world, h->scal_seq, dJ, dviol, h->stream, &h->launches);
    CUDA_TRY(h, cudaGetLastError());
    return DTO_OK;
}

extern "C" int dto_shard_scalars_dev(dto_handle* h, const double* dg, double* dJ, double* dviol) {
    if (!h || !dg || !dJ || !dviol) return DTO_ERR_INVALID;
    if (h->link_rank < 0 || h->P.batch != 1) {
        h->err = "dto_shard_scalars_dev: the shard is not linked";
        return DTO_ERR_INVALID;
    }
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (!h->d_scal_scratch) {
        void* p = nullptr;
        CUDA_TRY(h, cudaMalloc(&p, 2 * sizeof(unsigned long long)));
        h->allocs.push_back(p);
        CUDA_TRY(h, cudaMemset(p, 0, 2 * sizeof(unsigned long long)));  // synchronous: the kernel may run on either stream
        h->d_scal_scratch = (unsigned long long*)p;
    }
    ++h->scal_seq;
    // The residual (and, on the second stream, the objective) of the evaluation that was just enqueued are complete before
    // its Hessian assembler starts: the reduction and the exchange then run BESIDE the assembler, and the wait for the
    // slowest rank hides behind it.
    cudaStream_t st = h->stream;
    const bool beside = h->g_ready_valid && dg == h->g_ready_ptr && dJ == h->j_ready_ptr;
    if (beside) {
        CUDA_TRY(h, cudaStreamWaitEvent(h->aux_stream, h->ev_g_ready, 0));
        st = h->aux_stream;
    }
    h->g_ready_valid = false;
    launch_shard_scalars(h->xwin, h->d_peer_win, h->link_rank, h->link_world, h->scal_seq, h->P.n_cons_local, dg, h->d_row_is_eq,
                         h->d_scal_scratch, dJ, dviol, st, &h->launches);
    if (beside) {
        CUDA_TRY(h, cudaEventRecord(h->ev_scal_done, h->aux_stream));
        CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_scal_done, 0));
    }
    CUDA_TRY(h, cudaGetLastError());
    return DTO_OK;
}

// ---- instrumentation: device time of the interval kernels ------------------------------------------
extern "C" int dto_kernel_timing(dto_handle* h, int enable) {
    if (!h) return DTO_ERR_INVALID;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (enable && h->ev_pool.empty()) {
        h->ev_pool.resize(4096);
        for (auto& e : h->ev_pool) {
            CUDA_TRY(h, cudaEventCreate(&e.first));
            CUDA_TRY(h, cudaEventCreate(&e.second));
        }
    }
    h->timing = enable;
    h->ev_used = 0;
    h->k1_ms = 0.0;
    h->k1_count = 0;
    return DTO_OK;
}

extern "C" int dto_kernel_time_ms(dto_handle* h, double* ms_sum, int64_t* launches) {
    if (!h || !ms_sum || !launches) return DTO_ERR_INVALID;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (size_t i = 0; i < h->ev_used; ++i) {
        float ms = 0.f;
        CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev_pool[i].first, h->ev_pool[i].second));
        h->k1_ms += ms;
        h->k1_count += 1;
    }
    h->ev_used = 0;
    *ms_sum = h->k1_ms;
    *launches = h->k1_count;
    return DTO_OK;
}
