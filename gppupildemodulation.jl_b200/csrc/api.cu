// api.cu -- the C ABI of libgppd.so (include/gppd.h): handle, pipeline slots,
// host<->device staging and the launch sequence of one BATCH of tables.
//
// Launch sequence per batch (all on one stream, no host synchronisation inside):
//   [segmentation] -> basis -> [stats x2] -> harmonics -> harmonic fit
//                  -> direct fit of flagged fits -> demod -> export
// (method = direct: basis -> [stats] -> direct fit with HBM scratch -> demod -> export)
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <fcntl.h>
#include <functional>
#include <mutex>
#include <string>
#include <sys/stat.h>
#include <thread>
#include <unistd.h>
#include <vector>

#include <cuda.h>   // CUtensorMap and its enums only: the encoder is fetched through the runtime

#include "../../include/gppd.h"
#include "kernels.h"

using namespace gppd;

namespace {

thread_local std::string g_last_error;

#define CK(call)                                                                   \
    do {                                                                           \
        cudaError_t e_ = (call);                                                   \
        if (e_ != cudaSuccess) {                                                   \
            g_last_error = std::string(#call) + ": " + cudaGetErrorString(e_);     \
            return GPPD_ERR_CUDA;                                                  \
        }                                                                          \
    } while (0)

// GPPD_DEBUG_SYNC=1: synchronise after every pass and name the one that faulted
bool debug_sync() {
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("GPPD_DEBUG_SYNC");
        on = (e && *e && *e != '0') ? 1 : 0;
    }
    return on == 1;
}
#define DBG(stream, name)                                                          \
    do {                                                                           \
        if (debug_sync()) {                                                        \
            cudaError_t e_ = cudaStreamSynchronize(stream);                        \
            if (e_ == cudaSuccess) e_ = cudaGetLastError();                        \
            if (e_ != cudaSuccess) {                                               \
                g_last_error = std::string("pass ") + name + ": " + cudaGetErrorString(e_); \
                return GPPD_ERR_CUDA;                                              \
            }                                                                      \
        }                                                                          \
    } while (0)

// Buffers and events below free themselves: a Slot, a FileJob and the handle clean up by
// destruction, so that no buffer has to be remembered in a list to be released.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    int ensure(size_t bytes) {
        if (bytes <= cap) return GPPD_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            g_last_error = std::string("cudaMalloc: ") + cudaGetErrorString(e);
            p = nullptr;
            return GPPD_ERR_NOMEM;
        }
        cap = want;
        return GPPD_OK;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

#ifndef GPPD_NSLOTS
#define GPPD_NSLOTS 8
#endif
constexpr int NSLOTS = GPPD_NSLOTS;
constexpr int NPASS = GPPD_NPASS;
constexpr int MAX_TIMER = 1 << 16;

struct PassTimer {
    std::vector<cudaEvent_t> ev;      // begin/end pairs
    std::vector<int> pass;            // pass id per pair
    double ms[NPASS] = {0};
    long long count[NPASS] = {0};
    PassTimer() = default;
    PassTimer(const PassTimer &) = delete;
    PassTimer &operator=(const PassTimer &) = delete;
    ~PassTimer() {
        for (cudaEvent_t e : ev) cudaEventDestroy(e);
    }
};

// page-locked host buffer owned by the library (native file ingest)
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    PinBuf() = default;
    PinBuf(const PinBuf &) = delete;
    PinBuf &operator=(const PinBuf &) = delete;
    ~PinBuf() {
        if (p) cudaFreeHost(p);
    }
    int ensure(size_t bytes) {
        if (bytes <= cap) return GPPD_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        const size_t want = bytes + bytes / 8 + 4096;
        if (cudaMallocHost(&p, want) != cudaSuccess) {
            g_last_error = "cudaMallocHost failed";
            p = nullptr;
            return GPPD_ERR_NOMEM;
        }
        cap = want;
        return GPPD_OK;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// One file in flight on a slot (gppd_file_*).  stage: 0 free, 1 queued / being read and
// submitted, 2 results enqueued on the stream (gppd_file_wait can return), 3 being written.
struct FileJob {
    std::mutex m;
    std::condition_variable cv;
    int stage = 0;
    bool write_pending = false;
    int rc = GPPD_OK;
    std::string err;
    // the job as submitted (copied: the caller's buffers are not kept)
    std::string in_path;
    int64_t data_offset = 0, n = 0, row_bytes = 0, row_bytes_out = 0, time_off = 0, volt_off = 0, nfits = 0;
    double mjd = 0.0, window_s = 0.0;
    bool have_offsets = false, faint = false;
    double offsets[80];
    std::vector<double> timer1, timer2;
    gppd_options opt;
    PinBuf rows, rows_out, params, chi2, info, state;
};

struct Slot {
    cudaStream_t stream = nullptr;
    FileJob file;
    // staging of caller data (host-buffer entry points)
    DevBuf time, volt, volt_out, t, data, out, state_in, offsets, rows, rows_out;
    long long htab_vals = 0;        // values in htab after the last batch (test hook)
    DevBuf centres, cpart;          // --center empirical: [T][40] complex128 + partial sums
    int ncentres = 0;               // tables whose centres the last batch of this slot fitted
    // --center ellipse: descriptors, [T][40][6] maps + [T][40] statuses, partial sums, and the
    // complex128 arrays between the correction and the repack (t, corrected data, demodulated
    // out, FAINT states when the caller keeps none)
    DevBuf etabs, ell, estatus, epart, et, edata, eout, estate;
    int nellipses = 0;              // tables whose ellipses the last batch of this slot fitted
    DevBuf cov, covpart;            // GPPD_COVARIANCE: [nfits][36] + per-segment partial sums
    long long ncov = 0;             // fits whose covariances the last batch of this slot computed
    DevBuf params, chi2, info, trace, state_out;
    // batch scratch
    DevBuf state, basis, z, y, thkeys, nvalid, jobs, results;
    DevBuf spart1, spart2, partZ, partY, htab;
    DevBuf timers, lb, events, flags, tabs, exps, faintjobs, fbq, tmaps;
    PassTimer timer;
    cudaEvent_t fork = nullptr, join = nullptr;   // aux slots: hand-over to / from the main stream
};

}  // namespace

namespace {
// a few worker threads with a FIFO of closures (file readers / writers of one handle)
class IoPool {
  public:
    void start(int nthreads, int device) {
        std::lock_guard<std::mutex> lk(m_);
        if (!threads_.empty()) return;
        for (int i = 0; i < nthreads; ++i)
            threads_.emplace_back([this, device] {
                cudaSetDevice(device);
                for (;;) {
                    std::function<void()> f;
                    {
                        std::unique_lock<std::mutex> lk(m_);
                        cv_.wait(lk, [this] { return stop_ || !q_.empty(); });
                        if (q_.empty()) return;
                        f = std::move(q_.front());
                        q_.pop_front();
                    }
                    f();
                }
            });
    }
    void post(std::function<void()> f) {
        {
            std::lock_guard<std::mutex> lk(m_);
            q_.push_back(std::move(f));
        }
        cv_.notify_one();
    }
    ~IoPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
        }
        cv_.notify_all();
        for (std::thread &t : threads_) t.join();
    }

  private:
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<std::function<void()>> q_;
    std::vector<std::thread> threads_;
    bool stop_ = false;
};
}  // namespace

struct gppd_handle_s {
    int device = 0;
    bool timing = false;
    IoPool readers, writers;      // native file ingest / egress (started on first use)
    std::mutex launch_mutex;      // run_batch plans on the host: one planner at a time
    // FAINT and bright tables of a batch as two concurrent launch sequences (default on;
    // GPPD_SPLIT_CHAINS=0 or gppd_set_split_chains)
    bool split_chains = [] {
        const char *e = getenv("GPPD_SPLIT_CHAINS");
        return !(e && e[0] == '0');
    }();
    Slot slots[NSLOTS];
    // Second chain of each slot: the FAINT tables of a batch run on their own
    // (high-priority) stream, so that their latency-bound passes (segmentation,
    // statistics, fit) overlap the throughput-bound passes of the bright tables.
    Slot aux[NSLOTS];
    long long launches = 0;
};

namespace {

void fill_options(const gppd_options *o, FitOptions &f, int &method) {
    gppd_options d;
    memset(&d, 0, sizeof d);
    if (o) d = *o;
    f.flags = d.flags;
    f.maxfun = d.maxfun > 0 ? d.maxfun : 60;
    f.has_xinit = d.has_xinit;
    f.xinit[0] = d.xinit[0];
    f.xinit[1] = d.xinit[1];
    f.rhobeg = d.rhobeg > 0 ? d.rhobeg : 1.0;
    f.rhoend = d.rhoend > 0 ? d.rhoend : 1e-3;
    gppd_phirange(f.phi8);
    method = d.method;
    // the group mask travels in bits 16..23 of the kernels' flag word (GROUP_MASK_SHIFT)
    const unsigned mask = (d.group_mask & 0xffu) ? (d.group_mask & 0xffu) : 0xffu;
    f.flags = (f.flags & 0xffffu) | (mask << GROUP_MASK_SHIFT);
}

// CUtensorMap of one table of complex128 arrays, data[40][n] double2 seen as [40][2 n] doubles,
// box = 128 doubles (64 rows) x 40 channels.  cuTensorMapEncodeTiled is a driver entry point: it
// is fetched through the runtime, so that the library does not link libcuda.
static bool encode_array_map(CUtensorMap *out, const double2 *data, long long n) {
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static encode_fn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<encode_fn>(p);
        else
            cudaGetLastError();
    });
    if (!fn || n < 1 || 2 * (unsigned long long)n > 0x7fffffffull) return false;   // (int32 box coordinates)
    const cuuint64_t dims[2] = {2ull * (cuuint64_t)n, 40};
    const cuuint64_t strides[1] = {16ull * (cuuint64_t)n};        // bytes between channels
    const cuuint32_t box[2] = {128, 40}, estr[2] = {1, 1};       // 64 rows x 40 channels (harm_tc_kernels.cu: TC_ARR_ROWS)
    return fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double2 *>(data), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// cudaEvent pair around one pass (only when gppd_enable_timing is on)
struct PassScope {
    Slot *s;
    cudaStream_t st;
    bool on;
    PassScope(gppd_handle h, Slot &slot, cudaStream_t stream, int pass)
        : s(&slot), st(stream), on(h->timing) {
        if (!on) return;
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, st);
        s->timer.ev.push_back(a);
        s->timer.ev.push_back(b);
        s->timer.pass.push_back(pass);
    }
    ~PassScope() {
        if (on) cudaEventRecord(s->timer.ev.back(), st);
    }
};

// One table of a batch, as the entry points describe it (device pointers).
struct TableArgs {
    TableView tv{};
    OutView ov{};
    long long wrows = 0;            // <= 0 or >= n: whole table
    const int8_t *d_state_in = nullptr;
    const double *timer1 = nullptr, *timer2 = nullptr;  // HOST timers
    long long n1 = 0, n2 = 0, lag = 0;
    double pre = 0.0, post = 0.0;
    int8_t *d_state_out = nullptr;
    double *d_params = nullptr, *d_chi2 = nullptr;
    int *d_info = nullptr;
};

// Enqueue all passes of a batch on `stream`.  segment_only: stop after the
// segmentation (gppd_buildstates).
int run_batch(gppd_handle h, Slot &s, cudaStream_t stream, std::vector<TableArgs> &tabs,
              const gppd_options *opt, double *d_trace, bool segment_only) {
    FitOptions fo;
    int method;
    fill_options(opt, fo, method);
    // the covariance pass is an addition at the end of the sequence: the other passes see the
    // flag word they see without it
    const bool want_cov = (fo.flags & GPPD_COVARIANCE) != 0 && !segment_only;
    fo.flags &= ~GPPD_COVARIANCE;
    const int T = (int)tabs.size();
    if (T <= 0) return GPPD_OK;
    Launcher L{stream, &h->launches};
    int rc;

    // ---- plan ---------------------------------------------------------------
    long long R = 0, max_rows = 0, njobs_ll = 0, max_wrows = 0;
    int max_jobs = 0, max_timers = 0;
    size_t ntimers = 0, nlb = 0, nevents = 0;
    bool any_seg = false, any_state = false;
    std::vector<TableDesc> td(T);
    std::vector<ExportDesc> ex(T);
    std::vector<int> faint_jobs;   // jobs of the tables that have states
    for (int t = 0; t < T; ++t) {
        TableArgs &a = tabs[t];
        const long long n = a.tv.n;
        if (n < 2) {
            g_last_error = "need at least 2 rows";
            return GPPD_ERR_ARG;
        }
        const long long wrows = (a.wrows <= 0 || a.wrows >= n) ? n : a.wrows;
        const long long nj = (n + wrows - 1) / wrows;
        if (wrows > 0x7fffffffll || njobs_ll + nj > (0x7fffffffll / NDIODE)) {
            g_last_error = "too many windows / rows per window";
            return GPPD_ERR_ARG;
        }
        memset(&td[t], 0, sizeof(TableDesc));
        td[t].tv = a.tv;
        td[t].ov = a.ov;
        td[t].wrows = wrows;
        td[t].job0 = (int)njobs_ll;
        td[t].njobs = (int)nj;
        ex[t].fit0 = (int)njobs_ll * NDIODE;
        ex[t].nfits = (int)nj * NDIODE;
        ex[t].params = a.d_params;
        ex[t].chi2 = a.d_chi2;
        ex[t].info = a.d_info;
        const bool seg = !a.d_state_in && a.n1 > 0 && a.n2 > 0;
        if (seg) {
            if (a.n1 > MAX_TIMER || a.n2 > MAX_TIMER) {
                g_last_error = "timer series too long";
                return GPPD_ERR_ARG;
            }
            any_seg = true;
            ntimers += (size_t)(a.n1 + a.n2);
            nlb += (size_t)(a.n1 + a.n2 + 2);
            nevents += (size_t)(a.n1 + a.n2 + 1024);
            if (a.n1 + a.n2 > max_timers) max_timers = (int)(a.n1 + a.n2);
        }
        if (seg || a.d_state_in) {
            any_state = true;
            for (long long j = 0; j < nj; ++j) faint_jobs.push_back((int)(njobs_ll + j));
        }
        R += n;
        njobs_ll += nj;
        if (n > max_rows) max_rows = n;
        if (wrows > max_wrows) max_wrows = wrows;
        if (nj > max_jobs) max_jobs = (int)nj;
    }
    const int njobs = (int)njobs_ll, nfits = njobs * NDIODE, njg = njobs * NGROUP;
    const bool offs = (fo.flags & GPPD_FITOFFSETS) != 0;
    const bool empirical = (fo.flags & GPPD_CENTER_EMPIRICAL) != 0 && !segment_only;
    if (empirical && offs) {
        g_last_error = "GPPD_CENTER_EMPIRICAL and GPPD_FITOFFSETS exclude each other";
        return GPPD_ERR_ARG;
    }
    const bool direct = method == GPPD_METHOD_DIRECT;
    // the int8 tensor-core form of the harmonic sums takes dense METROLOGY tables (rows of
    // 80 floats, 16-byte aligned) and 16-byte aligned complex128 arrays; the other layouts
    // (strided FITS records before the unpack pass never get here) use the FP64 DMMA kernel.
    // GPPD_HARMONICS=dmma forces the DMMA kernel everywhere.
    bool dense = true;      // every table: rows of 80 floats back to back, 16-byte aligned
    for (int t = 0; t < T; ++t) {
        const TableView &v = td[t].tv;
        if (v.kind != 0 || (reinterpret_cast<unsigned long long>(v.volt) & 15ull) || v.volt_stride != 320)
            dense = false;
    }
    // ... and complex128 arrays (the demodulateall boundary), channel-major and 16-byte aligned
    bool arrays16 = true;
    for (int t = 0; t < T; ++t) {
        const TableView &v = td[t].tv;
        if (v.kind != 1 || (reinterpret_cast<unsigned long long>(v.data) & 15ull)) arrays16 = false;
    }
    // (a block of the tensor kernel serves all 8 groups and reads all 40 channels: measured on 1e8
    // rows, 18.1 ms with 8 groups and 15.4 ms with 4, against 3.7 ms per group for the per-group
    // DMMA kernel -- which therefore takes the calls with a partial mask of 4 groups or fewer)
    const int ngroups_on = __builtin_popcount((fo.flags >> GROUP_MASK_SHIFT) & 0xffu);
    const char *tmg = getenv("GPPD_TENSOR_MIN_GROUPS");
    const int min_groups = tmg ? atoi(tmg) : 5;
    int tensor = max_wrows < harm_tc_min_rows() ? 0 : (dense ? 1 : (arrays16 && ngroups_on >= min_groups ? 2 : 0));
    if (tensor == 2) {
        // one 2-D TMA descriptor per table: the kernel fetches 64 rows of all 40 channels with ONE
        // request (40 separate bulk copies per 32 rows measured 1 500 cycles of the SM's TMA unit)
        std::vector<CUtensorMap> tm((size_t)T);
        bool ok = s.tmaps.ensure(sizeof(CUtensorMap) * (size_t)T) == GPPD_OK;
        for (int t = 0; t < T && ok; ++t) ok = encode_array_map(&tm[t], td[t].tv.data, td[t].tv.n);
        if (ok) {
            CK(cudaMemcpyAsync(s.tmaps.p, tm.data(), sizeof(CUtensorMap) * (size_t)T, cudaMemcpyHostToDevice, stream));
            for (int t = 0; t < T; ++t) td[t].tmap = s.tmaps.as<CUtensorMap>() + t;
        } else {
            tensor = 0;         // (no encoder in this driver: the FP64 DMMA kernel)
        }
    }

    // partial sums are taken over FIXED row segments of each job (so that a fit's
    // result does not depend on the rest of the batch); P / SP = segments of the
    // longest job = grid width and stride of the partial buffers
    const int P = harm_max_segments(max_wrows);
    const int SP = stats_max_segments(max_wrows);
    if (P > 65535 || (long long)faint_jobs.size() * SP > 0x7fffffffll) {
        g_last_error = "job too long for one launch (more than 65 535 harmonic segments)";
        return GPPD_ERR_ARG;
    }

    // ---- scratch ------------------------------------------------------------
    if ((rc = s.tabs.ensure(sizeof(TableDesc) * (size_t)T))) return rc;
    if ((rc = s.exps.ensure(sizeof(ExportDesc) * (size_t)T))) return rc;
    if ((rc = s.basis.ensure(sizeof(double2) * (size_t)R))) return rc;
    if (any_seg) {
        if ((rc = s.state.ensure((size_t)R))) return rc;
        if ((rc = s.timers.ensure(sizeof(double) * ntimers))) return rc;
        if ((rc = s.lb.ensure(sizeof(long long) * nlb))) return rc;
        if ((rc = s.events.ensure((size_t)SEG_EVENT_BYTES * nevents))) return rc;
        if ((rc = s.flags.ensure(2 * sizeof(int) * (size_t)T))) return rc;
    }
    if (!segment_only) {
        if ((rc = s.thkeys.ensure(sizeof(unsigned long long) * 2 * (size_t)njobs))) return rc;
        if ((rc = s.nvalid.ensure(sizeof(int) * 5 * (size_t)njobs))) return rc;
        if ((rc = s.jobs.ensure(sizeof(JobInfo) * (size_t)njobs))) return rc;
        if ((rc = s.results.ensure(sizeof(FitResult) * (size_t)nfits))) return rc;
        if (any_state) {
            if ((rc = s.spart1.ensure(sizeof(double) * STATS_VALS * (size_t)njg * SP))) return rc;
            if ((rc = s.spart2.ensure(sizeof(double) * 32 * (size_t)njg))) return rc;
            if ((rc = s.faintjobs.ensure(sizeof(int) * faint_jobs.size()))) return rc;
        }
        if (direct) {
            if ((rc = s.z.ensure(sizeof(double2) * (size_t)R * NDIODE))) return rc;
            if (offs)
                if ((rc = s.y.ensure(sizeof(double2) * (size_t)R * NDIODE))) return rc;
        } else {
            if ((rc = s.partZ.ensure(sizeof(double) * HP_Z * 4 * (size_t)njg * P))) return rc;
            if (offs)
                if ((rc = s.partY.ensure(sizeof(double) * HP_Y * 4 * (size_t)njg * P))) return rc;
            if ((rc = s.htab.ensure(sizeof(double) * HV_COUNT * (size_t)nfits))) return rc;
            if ((rc = s.fbq.ensure(sizeof(int) * ((size_t)nfits + 1)))) return rc;
        }
    }

    const int CP = want_cov ? cov_max_segments(max_wrows) : 0;
    if (want_cov) {
        if (CP > 65535) {
            g_last_error = "job too long for one launch (more than 65 535 covariance segments)";
            return GPPD_ERR_ARG;
        }
        if ((rc = s.cov.ensure(sizeof(double) * GPPD_COV_STRIDE * (size_t)nfits))) return rc;
        if ((rc = s.covpart.ensure(sizeof(double) * COV_VALS * NDIODE * (size_t)njobs * CP))) return rc;
    }

    s.ncentres = 0;
    if (!segment_only) {
        s.nellipses = 0;
        s.ncov = 0;
    }
    if (empirical) {
        // offsets === true: every table gets its own 40 centres, fitted on the device
        if ((rc = s.centres.ensure(sizeof(double2) * NCHAN * (size_t)T))) return rc;
        if ((rc = s.cpart.ensure(sizeof(double) * CIRC_VALS * NCHAN * (size_t)T *
                                 circle_max_segments(max_rows))))
            return rc;
        for (int t = 0; t < T; ++t) {
            if (td[t].tv.kind != 0) {
                g_last_error = "GPPD_CENTER_EMPIRICAL applies to METROLOGY tables only";
                return GPPD_ERR_ARG;
            }
            td[t].tv.offsets = s.centres.as<double2>() + (size_t)t * NCHAN;
        }
        s.ncentres = T;
    }

    // ---- carve per-table slices, upload descriptors ---------------------------
    {
        size_t row_off = 0, tim_off = 0, lb_off = 0, ev_off = 0;
        for (int t = 0; t < T; ++t) {
            TableArgs &a = tabs[t];
            TableDesc &d = td[t];
            const long long n = a.tv.n;
            d.basis = s.basis.as<double2>() + row_off;
            if (direct && !segment_only) {
                d.z = s.z.as<double2>() + row_off * NDIODE;
                d.y = offs ? s.y.as<double2>() + row_off * NDIODE : nullptr;
            }
            const bool seg = !a.d_state_in && a.n1 > 0 && a.n2 > 0;
            if (seg) {
                d.state = a.d_state_out ? a.d_state_out : s.state.as<int8_t>() + row_off;
                d.seg.timer1 = s.timers.as<double>() + tim_off;
                d.seg.timer2 = d.seg.timer1 + a.n1;
                d.seg.n1 = (int)a.n1;
                d.seg.n2 = (int)a.n2;
                d.seg.lag = a.lag;
                d.seg.pre = a.pre;
                d.seg.post = a.post;
                d.seg.lb = s.lb.as<long long>() + lb_off;
                d.seg.events = s.events.as<char>() + ev_off * SEG_EVENT_BYTES;
                d.seg.max_events = (int)(a.n1 + a.n2 + 1024);
                d.seg.flags = s.flags.as<int>() + 2 * t;
                // small pageable copies are staged by the runtime before returning
                CK(cudaMemcpyAsync((void *)d.seg.timer1, a.timer1, sizeof(double) * (size_t)a.n1,
                                   cudaMemcpyHostToDevice, stream));
                CK(cudaMemcpyAsync((void *)d.seg.timer2, a.timer2, sizeof(double) * (size_t)a.n2,
                                   cudaMemcpyHostToDevice, stream));
                tim_off += (size_t)(a.n1 + a.n2);
                lb_off += (size_t)(a.n1 + a.n2 + 2);
                ev_off += (size_t)(a.n1 + a.n2 + 1024);
            } else if (a.d_state_in) {
                d.state = const_cast<int8_t *>(a.d_state_in);
                if (a.d_state_out && a.d_state_out != a.d_state_in)
                    CK(cudaMemcpyAsync(a.d_state_out, a.d_state_in, (size_t)n,
                                       cudaMemcpyDeviceToDevice, stream));
            }
            row_off += (size_t)n;
        }
        CK(cudaMemcpyAsync(s.tabs.p, td.data(), sizeof(TableDesc) * (size_t)T,
                           cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(s.exps.p, ex.data(), sizeof(ExportDesc) * (size_t)T,
                           cudaMemcpyHostToDevice, stream));
        if (any_state && !segment_only)
            CK(cudaMemcpyAsync(s.faintjobs.p, faint_jobs.data(), sizeof(int) * faint_jobs.size(),
                               cudaMemcpyHostToDevice, stream));
    }
    const TableDesc *d_tabs = s.tabs.as<TableDesc>();

    // ---- launch sequence ------------------------------------------------------
    if (any_seg) {
        PassScope ps(h, s, stream, GPPD_PASS_SEGMENT);
        launch_segmentation(L, d_tabs, T, max_rows, max_timers);
    }
    DBG(stream, "segmentation");
    if (segment_only) {
        CK(cudaGetLastError());
        return GPPD_OK;
    }
    if (empirical) {
        PassScope ps(h, s, stream, GPPD_PASS_BASIS);
        launch_circle(L, d_tabs, T, max_rows, s.cpart.as<double>());
    }
    DBG(stream, "centres");
    {
        PassScope ps(h, s, stream, GPPD_PASS_BASIS);
        launch_basis(L, d_tabs, T, max_rows, max_jobs, njobs, fo.flags,
                     s.thkeys.as<unsigned long long>(), s.nvalid.as<int>(), s.jobs.as<JobInfo>());
    }
    DBG(stream, "basis");
    if (any_state) {
        PassScope ps(h, s, stream, GPPD_PASS_STATS);
        launch_stats(L, d_tabs, s.jobs.as<JobInfo>(), njobs, s.faintjobs.as<int>(),
                     (int)faint_jobs.size(), s.nvalid.as<int>(), fo.flags, SP, s.spart1.as<double>(),
                     s.spart2.as<double>(), dense && !getenv("GPPD_STATS_PLAIN"));
    }
    DBG(stream, "stats");
    if (direct) {
        PassScope ps(h, s, stream, GPPD_PASS_FIT);
        launch_fit_direct(L, d_tabs, s.jobs.as<JobInfo>(), nfits, SP, s.spart1.as<double>(),
                          s.spart2.as<double>(), fo, true, s.results.as<FitResult>(), d_trace, nullptr);
    } else {
        {
            PassScope ps(h, s, stream, GPPD_PASS_HARMONICS);
            launch_harmonics(L, d_tabs, s.jobs.as<JobInfo>(), njobs, fo.flags, P, SP,
                             s.spart1.as<double>(), s.spart2.as<double>(), s.partZ.as<double>(),
                             s.partY.as<double>(), s.htab.as<double>(), tensor);
            s.htab_vals = (long long)nfits * (offs ? HV_COUNT : HV_Y0R);
        }
        DBG(stream, "harmonics");
        {
            PassScope ps(h, s, stream, GPPD_PASS_FIT);
            CK(cudaMemsetAsync(s.fbq.p, 0, sizeof(int), stream));
            launch_fit_harmonic(L, d_tabs, s.jobs.as<JobInfo>(), s.htab.as<double>(), nfits, fo,
                                s.results.as<FitResult>(), d_trace, s.fbq.as<int>());
        }
        DBG(stream, "fit_harmonic");
        {
            PassScope ps(h, s, stream, GPPD_PASS_FALLBACK);
            launch_fit_direct(L, d_tabs, s.jobs.as<JobInfo>(), nfits, SP, s.spart1.as<double>(),
                              s.spart2.as<double>(), fo, false, s.results.as<FitResult>(), d_trace,
                              s.fbq.as<int>());
        }
    }
    DBG(stream, "fit_direct");
    {
        PassScope ps(h, s, stream, GPPD_PASS_DEMOD);
        bool arrays = true;
        for (int t = 0; t < T; ++t) arrays = arrays && td[t].tv.kind == 1 && td[t].ov.kind == 1;
        launch_demod(L, d_tabs, T, max_rows, s.results.as<FitResult>(), fo.flags, arrays);
    }
    DBG(stream, "demod");
    if (want_cov) {
        PassScope ps(h, s, stream, GPPD_PASS_EXPORT);
        launch_covariance(L, d_tabs, s.jobs.as<JobInfo>(), njobs, s.results.as<FitResult>(),
                          any_state ? s.spart2.as<double>() : nullptr, fo.flags, CP, s.covpart.as<double>(),
                          s.cov.as<double>());
        s.ncov = nfits;
    }
    DBG(stream, "covariance");
    {
        PassScope ps(h, s, stream, GPPD_PASS_EXPORT);
        launch_export(L, s.exps.as<ExportDesc>(), T, max_jobs * NDIODE, s.results.as<FitResult>(), fo.flags);
    }
    DBG(stream, "export");
    CK(cudaGetLastError());
    return GPPD_OK;
}

int check_handle(gppd_handle h) {
    if (!h) {
        g_last_error = "null handle";
        return GPPD_ERR_ARG;
    }
    CK(cudaSetDevice(h->device));
    return GPPD_OK;
}

// The options of a table entry point: the caller's (or zeros) with the centre mode applied,
// after the rejection of every combination that no table path runs.  The centre mode is the
// offsets of processmetrology (src/GPPupilDemodulation.jl:150-157): a vector => subtract it;
// true (GPPD_CENTER_EMPIRICAL) => circle centres fitted here; false (NULL) => fitoffsets.
// GPPD_CENTER_ELLIPSE ignores the vector.
int table_options(const gppd_options *opt, bool have_offsets, gppd_options &o) {
    memset(&o, 0, sizeof o);
    if (opt) o = *opt;
    if ((o.flags & GPPD_CENTER_ELLIPSE) && (o.flags & (GPPD_CENTER_EMPIRICAL | GPPD_FITOFFSETS))) {
        g_last_error = "GPPD_CENTER_ELLIPSE excludes GPPD_CENTER_EMPIRICAL and GPPD_FITOFFSETS";
        return GPPD_ERR_ARG;
    }
    if ((o.group_mask & 0xffu) != 0 && (o.group_mask & 0xffu) != 0xffu) {
        g_last_error = "gppd_options.group_mask: a partial mask applies to the demodulate_f64 entry points only";
        return GPPD_ERR_UNSUPPORTED;
    }
    if (!(o.flags & (GPPD_CENTER_EMPIRICAL | GPPD_CENTER_ELLIPSE)) && !have_offsets) o.flags |= GPPD_FITOFFSETS;
    else o.flags &= ~GPPD_FITOFFSETS;
    return GPPD_OK;
}

// The options of the array entry points: GPPD_CENTER_ELLIPSE corrects METROLOGY tables only.
int check_array_options(const gppd_options *opt) {
    if (opt && (opt->flags & GPPD_CENTER_ELLIPSE)) {
        g_last_error = "GPPD_CENTER_ELLIPSE applies to the table entry points only";
        return GPPD_ERR_UNSUPPORTED;
    }
    return GPPD_OK;
}

void table_views(int64_t n, double mjd, const int32_t *d_time, const float *d_volt,
                 const double *d_offsets, float *d_volt_out, uint32_t flags, TableArgs &a) {
    a.tv.kind = 0;
    a.tv.big_endian = (flags & GPPD_BIG_ENDIAN) ? 1 : 0;
    a.tv.n = n;
    a.tv.time_us = d_time;
    a.tv.time_stride = 4;
    a.tv.volt = d_volt;
    a.tv.volt_stride = 320;
    a.tv.tmjd = 86400.0 * mjd;   // DAY_TO_SEC * mjd
    a.tv.offsets = reinterpret_cast<const double2 *>(d_offsets);
    a.ov.kind = 0;
    a.ov.big_endian = a.tv.big_endian;
    a.ov.keepraw = (flags & GPPD_KEEPRAW) ? 1 : 0;
    a.ov.volt = d_volt_out;
    a.ov.volt_stride = a.ov.keepraw ? 576 : 320;
}

// the complex128-array counterpart (the demodulateall boundary): t[n], data[40][n] -> out[40][n]
void array_views(int64_t n, const double *d_t, const double2 *d_data, double2 *d_out, TableArgs &a) {
    a.tv.kind = 1;
    a.tv.n = n;
    a.tv.t = d_t;
    a.tv.data = d_data;
    a.ov.kind = 1;
    a.ov.out = d_out;
}

// `--center ellipse` on a batch of kind-0 tables: a composition of existing passes around the
// ellipse kernels (centre_kernels.cu), all on `stream`:
//   1. FAINT segmentation of the tables that have timers (run_batch, segment_only)
//   2. moments + conic solve per channel -> s.ell / s.estatus      (GPPD_PASS_BASIS)
//   3. the correction: TIME + VOLT rows -> t, data[40][n] complex128 (GPPD_PASS_BASIS)
//   4. the array path of gppd_demodulate_f64_dev on (t, data, states) -> out[40][n]
//   5. the repack of out into the caller's VOLT rows               (GPPD_PASS_DEMOD)
int run_batch_ellipse(gppd_handle h, Slot &s, cudaStream_t stream, std::vector<TableArgs> &tabs,
                      const gppd_options &o) {
    const int T = (int)tabs.size();
    if (T <= 0) return GPPD_OK;
    long long R = 0, max_rows = 0, R_state = 0;
    for (const TableArgs &a : tabs) {
        if (a.tv.kind != 0 || a.tv.n < 2) {
            g_last_error = "GPPD_CENTER_ELLIPSE: need METROLOGY tables of at least 2 rows";
            return GPPD_ERR_ARG;
        }
        R += a.tv.n;
        if (a.tv.n > max_rows) max_rows = a.tv.n;
        if (a.n1 > 0 && a.n2 > 0 && !a.d_state_out) R_state += a.tv.n;
    }
    const int P = circle_max_segments(max_rows);
    int rc;
    if ((rc = s.etabs.ensure(sizeof(TableDesc) * (size_t)T))) return rc;
    if ((rc = s.ell.ensure(sizeof(double) * ELL_STRIDE * NCHAN * (size_t)T))) return rc;
    if ((rc = s.estatus.ensure(sizeof(int) * NCHAN * (size_t)T))) return rc;
    if ((rc = s.epart.ensure(sizeof(double) * ELL_VALS * NCHAN * (size_t)T * (size_t)P))) return rc;
    if ((rc = s.et.ensure(sizeof(double) * (size_t)R))) return rc;
    if ((rc = s.edata.ensure(sizeof(double2) * NCHAN * (size_t)R))) return rc;
    if ((rc = s.eout.ensure(sizeof(double2) * NCHAN * (size_t)R))) return rc;
    if (R_state)
        if ((rc = s.estate.ensure((size_t)R_state))) return rc;

    // 1. states of the FAINT tables (into the caller's buffer when there is one)
    std::vector<TableArgs> seg;
    std::vector<int8_t *> states((size_t)T, nullptr);
    {
        size_t st_off = 0;
        for (int t = 0; t < T; ++t) {
            TableArgs &a = tabs[t];
            if (!(a.n1 > 0 && a.n2 > 0)) continue;
            if (!a.d_state_out) {
                a.d_state_out = s.estate.as<int8_t>() + st_off;
                st_off += (size_t)a.tv.n;
            }
            states[t] = a.d_state_out;
            seg.push_back(a);
        }
    }
    if (!seg.empty())
        if ((rc = run_batch(h, s, stream, seg, nullptr, nullptr, true))) return rc;

    // 2. + 3. the ellipses and the corrected arrays
    std::vector<TableDesc> td((size_t)T);
    std::vector<TableArgs> arr((size_t)T);
    {
        size_t row_off = 0;
        for (int t = 0; t < T; ++t) {
            const TableArgs &a = tabs[t];
            TableDesc &d = td[t];
            memset(&d, 0, sizeof d);
            d.tv = a.tv;
            d.ov = a.ov;
            d.tv.offsets = reinterpret_cast<const double2 *>(s.ell.as<double>() + (size_t)t * NCHAN * ELL_STRIDE);
            d.tv.t = s.et.as<double>() + row_off;
            d.tv.data = s.edata.as<double2>() + NCHAN * row_off;
            d.ov.out = s.eout.as<double2>() + NCHAN * row_off;
            d.state = states[t];
            TableArgs &b = arr[t];
            array_views(a.tv.n, d.tv.t, d.tv.data, d.ov.out, b);
            b.wrows = a.wrows;
            b.d_state_in = states[t];
            b.d_params = a.d_params;
            b.d_chi2 = a.d_chi2;
            b.d_info = a.d_info;
            row_off += (size_t)a.tv.n;
        }
    }
    // (small pageable copy: staged by the runtime before cudaMemcpyAsync returns)
    CK(cudaMemcpyAsync(s.etabs.p, td.data(), sizeof(TableDesc) * (size_t)T, cudaMemcpyHostToDevice, stream));
    const TableDesc *d_tabs = s.etabs.as<TableDesc>();
    Launcher L{stream, &h->launches};
    {
        PassScope ps(h, s, stream, GPPD_PASS_BASIS);
        launch_ellipse_fit(L, d_tabs, T, max_rows, s.epart.as<double>(), s.ell.as<double>(), s.estatus.as<int>());
        launch_ellipse_apply(L, d_tabs, T, max_rows, s.ell.as<double>());
    }
    DBG(stream, "ellipse");

    // 4. the ordinary array path, NoOffsets model (GPPD_FP32 has no array form: no effect here)
    gppd_options o4 = o;
    o4.flags &= ~(GPPD_CENTER_ELLIPSE | GPPD_KEEPRAW | GPPD_BIG_ENDIAN | GPPD_FP32);
    if ((rc = run_batch(h, s, stream, arr, &o4, nullptr, false))) return rc;

    // 5. back to VOLT rows
    {
        PassScope ps(h, s, stream, GPPD_PASS_DEMOD);
        launch_repack_arrays(L, d_tabs, T, max_rows, (o.flags & GPPD_KEEPRAW) != 0);
    }
    DBG(stream, "repack");
    CK(cudaGetLastError());
    s.nellipses = T;
    return GPPD_OK;
}

// The batch of a table entry point on slot `slot`, with options from table_options: the ellipse
// composition, the FAINT and the bright tables as two concurrent chains (the FAINT one on the
// slot's aux stream), or one launch sequence.  Results do not depend on the batching: all
// partial sums are over fixed row segments.
int run_tables(gppd_handle h, int slot, cudaStream_t stream, std::vector<TableArgs> &tabs,
               const gppd_options &o) {
    Slot &s = h->slots[slot];
    if (o.flags & GPPD_CENTER_ELLIPSE) return run_batch_ellipse(h, s, stream, tabs, o);
    std::vector<TableArgs> faint, bright;
    for (TableArgs &a : tabs) (a.n1 > 0 ? faint : bright).push_back(a);
    // (the fit's latency-bound tail and the HBM-bound demodulation of one chain overlap the
    // issue-bound harmonic pass of the other: measured +8 % on the 100-table night.  Each
    // pass is then two launches per batch; gppd_pass_times adds their durations.
    // GPPD_SPLIT_CHAINS=0 or gppd_set_split_chains(h, 0) keeps one launch sequence.)
    // (not for batches of very many small fits: there the one-thread-per-fit solver dominates
    // and two concurrent launches of it are slower than one -- measured, 20 tables: 5 000-row
    // windows (12 800 fits) 3.3 against 4.3 ms, 2 000-row windows (32 000 fits) 5.0 against 4.3)
    long long nfits_total = 0;
    for (const TableArgs &a : tabs) {
        const long long w = (a.wrows <= 0 || a.wrows >= a.tv.n) ? a.tv.n : a.wrows;
        nfits_total += (a.tv.n + w - 1) / w * NDIODE;
    }
    // (with GPPD_COVARIANCE too: every fit's covariance then lands on the slot gppd_covariances reads)
    if (faint.empty() || bright.empty() || !h->split_chains || nfits_total > 16384 ||
        (o.flags & (GPPD_CENTER_EMPIRICAL | GPPD_COVARIANCE)))
        return run_batch(h, s, stream, tabs, &o, nullptr, false);
    Slot &sb = h->aux[slot];
    int rc;
    CK(cudaEventRecord(sb.fork, stream));
    CK(cudaStreamWaitEvent(sb.stream, sb.fork, 0));
    if ((rc = run_batch(h, sb, sb.stream, faint, &o, nullptr, false))) return rc;
    if ((rc = run_batch(h, s, stream, bright, &o, nullptr, false))) return rc;
    CK(cudaEventRecord(sb.join, sb.stream));
    CK(cudaStreamWaitEvent(stream, sb.join, 0));
    return GPPD_OK;
}

// Rows per window and number of windows of a table of FITS records: gppd_table_windows on the
// TIME of the first two records, read big-endian on the host (src/GPPupilDemodulation.jl:192),
// once TIME and VOLT are known to lie inside the record without overlapping.
int record_windows(int64_t n, const unsigned char *rows, int64_t row_bytes, int64_t time_off, int64_t volt_off,
                   double mjd, double window_s, int64_t &wrows, int64_t &nwin) {
    if (time_off < 0 || volt_off < 0 || time_off + 4 > row_bytes || volt_off + 320 > row_bytes ||
        (time_off + 4 > volt_off && time_off < volt_off + 320)) {
        g_last_error = "fits rows: TIME or VOLT outside the record";
        return GPPD_ERR_ARG;
    }
    int32_t t01[2];
    for (int k = 0; k < 2; ++k) {
        const unsigned char *p = rows + k * row_bytes + time_off;
        t01[k] = (int32_t)(((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]);
    }
    return gppd_table_windows(n, t01, mjd, window_s, &wrows, &nwin);
}

// One table of a host-buffer entry point, enqueued on the stream of slot `slot`.  The table is
// either TIME + VOLT arrays (`rows` null) or FITS records (`rows`: big-endian, `row_bytes`
// apart, TIME at `time_off` and VOLT at `volt_off`; already in s.rows when `rows_uploaded`).
// `out` receives VOLT rows in the form of the input: arrays, or records with VOLT replaced.
int stage_table(gppd_handle h, int slot, int64_t n, const int32_t *time_us, const float *volt, const void *rows,
                bool rows_uploaded, int64_t row_bytes, int64_t time_off, int64_t volt_off, double mjd,
                const double *offsets, const double *timer1, int64_t n1, const double *timer2, int64_t n2,
                double window_s, const gppd_options *opt, void *out, double *params, double *chi2,
                int32_t *info, int8_t *state_out) {
    const bool recs = rows != nullptr;
    int64_t wrows = n, nwin = 1;
    int rc = recs ? record_windows(n, reinterpret_cast<const unsigned char *>(rows), row_bytes, time_off,
                                   volt_off, mjd, window_s, wrows, nwin)
                  : gppd_table_windows(n, time_us, mjd, window_s, &wrows, &nwin);
    if (rc) return rc;
    gppd_options o;
    if ((rc = table_options(opt, offsets != nullptr, o))) return rc;
    if (recs) o.flags &= ~GPPD_BIG_ENDIAN;    // the unpack pass delivers little-endian arrays
    const int out_floats = (o.flags & GPPD_KEEPRAW) ? 144 : 80;
    const int64_t row_bytes_out = row_bytes + 4 * (out_floats - 80);
    const size_t nfits = (size_t)nwin * NDIODE;
    const size_t vbytes = sizeof(float) * 80 * (size_t)n, obytes = sizeof(float) * out_floats * (size_t)n;
    Slot &s = h->slots[slot];
    cudaStream_t st = s.stream;
    if (!rows_uploaded) CK(cudaStreamSynchronize(st));  // slot reuse: previous table of this slot must be done
    std::lock_guard<std::mutex> lk(h->launch_mutex);
    if (recs) {
        if ((rc = s.rows.ensure((size_t)n * (size_t)row_bytes))) return rc;
        if ((rc = s.rows_out.ensure((size_t)n * (size_t)row_bytes_out))) return rc;
    }
    if ((rc = s.time.ensure(sizeof(int32_t) * (size_t)n))) return rc;
    if ((rc = s.volt.ensure(vbytes))) return rc;
    if ((rc = s.volt_out.ensure(obytes))) return rc;
    if ((rc = s.params.ensure(sizeof(double) * 6 * nfits))) return rc;
    if ((rc = s.chi2.ensure(sizeof(double) * nfits))) return rc;
    if ((rc = s.info.ensure(sizeof(int) * GPPD_INFO_STRIDE * nfits))) return rc;
    if ((rc = s.state_out.ensure((size_t)n))) return rc;
    if ((rc = s.offsets.ensure(sizeof(double) * 80))) return rc;
    if (!recs) {
        CK(cudaMemcpyAsync(s.time.p, time_us, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(s.volt.p, volt, vbytes, cudaMemcpyHostToDevice, st));
    } else if (!rows_uploaded) {
        CK(cudaMemcpyAsync(s.rows.p, rows, (size_t)n * (size_t)row_bytes, cudaMemcpyHostToDevice, st));
    }
    if (offsets)
        CK(cudaMemcpyAsync(s.offsets.p, offsets, sizeof(double) * 80, cudaMemcpyHostToDevice, st));
    Launcher L{st, &h->launches};
    if (recs)
        launch_unpack_rows(L, s.rows.p, n, row_bytes, time_off, volt_off, s.time.as<int32_t>(), s.volt.as<float>());
    std::vector<TableArgs> tabs(1);
    TableArgs &a = tabs[0];
    table_views(n, mjd, s.time.as<int32_t>(), s.volt.as<float>(),
                offsets ? s.offsets.as<double>() : nullptr, s.volt_out.as<float>(), o.flags, a);
    a.wrows = wrows;
    const bool faint = timer1 && timer2 && n1 > 0 && n2 > 0;
    a.timer1 = timer1;
    a.timer2 = timer2;
    a.n1 = faint ? n1 : 0;
    a.n2 = faint ? n2 : 0;
    a.d_params = s.params.as<double>();
    a.d_chi2 = s.chi2.as<double>();
    a.d_info = s.info.as<int>();
    a.d_state_out = s.state_out.as<int8_t>();
    if ((rc = run_tables(h, slot, st, tabs, o))) return rc;
    if (recs) {
        launch_pack_rows(L, s.rows.p, n, row_bytes, volt_off, s.volt_out.as<float>(), out_floats, s.rows_out.p,
                         row_bytes_out);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out, s.rows_out.p, (size_t)n * (size_t)row_bytes_out, cudaMemcpyDeviceToHost, st));
    } else {
        CK(cudaMemcpyAsync(out, s.volt_out.p, obytes, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaMemcpyAsync(params, s.params.p, sizeof(double) * 6 * nfits, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(chi2, s.chi2.p, sizeof(double) * nfits, cudaMemcpyDeviceToHost, st));
    if (info)
        CK(cudaMemcpyAsync(info, s.info.p, sizeof(int) * GPPD_INFO_STRIDE * nfits, cudaMemcpyDeviceToHost, st));
    if (state_out && faint)
        CK(cudaMemcpyAsync(state_out, s.state_out.p, (size_t)n, cudaMemcpyDeviceToHost, st));
    return GPPD_OK;
}

}  // namespace

// ===========================================================================
extern "C" {

int gppd_version(void) { return GPPD_VERSION; }

const char *gppd_strerror(int status) {
    switch (status) {
    case GPPD_OK: return "ok";
    case GPPD_ERR_ARG: return "bad argument";
    case GPPD_ERR_CUDA: return "CUDA error";
    case GPPD_ERR_NO_DEVICE: return "no sm_100 CUDA device (libgppd has no CPU fallback)";
    case GPPD_ERR_NOMEM: return "out of device memory";
    case GPPD_ERR_UNSUPPORTED: return "unsupported";
    default: return "unknown status";
    }
}

const char *gppd_last_error(void) { return g_last_error.c_str(); }

int gppd_idx(int side, int telescope, int diode) {
    if ((side != 0 && side != 16) || telescope < 1 || telescope > 4 || diode < 1 || diode > 5)
        return -1;
    if (diode == 5) return 32 + side / 4 + (telescope - 1) + 1;
    return side + (diode - 1) + (telescope - 1) * 4 + 1;
}

int gppd_phirange(double *phi8) {
    if (!phi8) return GPPD_ERR_ARG;
    // Julia's range(-pi, pi, 8) is evaluated in twice precision: each element is
    // the correctly rounded -pi_f + k (2 pi_f / 7); long double reproduces it.
    const long double lo = -(long double)PI_F64, hi = (long double)PI_F64;
    for (int k = 0; k < 8; ++k)
        phi8[k] = (double)(((long double)(7 - k) * lo + (long double)k * hi) / 7.0L);
    phi8[0] = -PI_F64;
    phi8[7] = PI_F64;
    return GPPD_OK;
}

int gppd_create(int device, gppd_handle *out) {
    if (!out) return GPPD_ERR_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        g_last_error = e != cudaSuccess ? cudaGetErrorString(e) : "no such CUDA device";
        return GPPD_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        g_last_error = std::string("device is sm_") + std::to_string(prop.major) +
                       std::to_string(prop.minor) + ", libgppd is built for sm_100a only";
        return GPPD_ERR_NO_DEVICE;
    }
    CK(cudaSetDevice(device));
    gppd_handle h = new gppd_handle_s;
    h->device = device;
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    for (int i = 0; i < NSLOTS; ++i) {
        cudaError_t es = cudaStreamCreateWithFlags(&h->slots[i].stream, cudaStreamNonBlocking);
        if (es == cudaSuccess)
            es = cudaStreamCreateWithPriority(&h->aux[i].stream, cudaStreamNonBlocking, prio_greatest);
        if (es == cudaSuccess) es = cudaEventCreateWithFlags(&h->aux[i].fork, cudaEventDisableTiming);
        if (es == cudaSuccess) es = cudaEventCreateWithFlags(&h->aux[i].join, cudaEventDisableTiming);
        if (es != cudaSuccess) {
            g_last_error = cudaGetErrorString(es);
            gppd_destroy(h);
            return GPPD_ERR_CUDA;
        }
    }
    *out = h;
    return GPPD_OK;
}

int gppd_destroy(gppd_handle h) {
    if (!h) return GPPD_OK;
    cudaSetDevice(h->device);
    gppd_file_drain(h);
    for (int i = 0; i < 2 * NSLOTS; ++i) {
        Slot &s = i < NSLOTS ? h->slots[i] : h->aux[i - NSLOTS];
        if (s.stream) {
            cudaStreamSynchronize(s.stream);
            cudaStreamDestroy(s.stream);
        }
        if (s.fork) cudaEventDestroy(s.fork);
        if (s.join) cudaEventDestroy(s.join);
    }
    delete h;   // (the slots' buffers and pass timers free themselves, on the handle's device)
    return GPPD_OK;
}

int gppd_alloc_pinned(gppd_handle h, uint64_t bytes, void **out) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (!out) return GPPD_ERR_ARG;
    CK(cudaMallocHost(out, bytes ? bytes : 1));
    return GPPD_OK;
}

int gppd_free_pinned(gppd_handle h, void *p) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (p) CK(cudaFreeHost(p));
    return GPPD_OK;
}

int gppd_num_slots(gppd_handle) { return NSLOTS; }

int gppd_centres(gppd_handle h, int slot, int64_t ntables, double *centres) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !centres || ntables < 1) return GPPD_ERR_ARG;
    Slot &s = h->slots[slot];
    if (ntables > s.ncentres) {
        g_last_error = "centres: the last call on this slot fitted fewer tables' centres";
        return GPPD_ERR_ARG;
    }
    CK(cudaStreamSynchronize(s.stream));
    CK(cudaMemcpy(centres, s.centres.p, sizeof(double2) * NCHAN * (size_t)ntables,
                  cudaMemcpyDeviceToHost));
    return GPPD_OK;
}

int gppd_ellipses(gppd_handle h, int slot, int64_t ntables, double *ell, int32_t *status) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !ell || ntables < 1) return GPPD_ERR_ARG;
    Slot &s = h->slots[slot];
    if (ntables > s.nellipses) {
        g_last_error = "ellipses: the last call on this slot fitted fewer tables' ellipses";
        return GPPD_ERR_ARG;
    }
    CK(cudaStreamSynchronize(s.stream));
    CK(cudaMemcpy(ell, s.ell.p, sizeof(double) * GPPD_ELLIPSE_STRIDE * NCHAN * (size_t)ntables,
                  cudaMemcpyDeviceToHost));
    if (status)
        CK(cudaMemcpy(status, s.estatus.p, sizeof(int32_t) * NCHAN * (size_t)ntables, cudaMemcpyDeviceToHost));
    return GPPD_OK;
}

int gppd_covariances(gppd_handle h, int slot, int64_t nfits, double *cov) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !cov || nfits < 1) return GPPD_ERR_ARG;
    Slot &s = h->slots[slot];
    if (nfits > s.ncov) {
        g_last_error = "covariances: the last call on this slot ran without GPPD_COVARIANCE or had fewer fits";
        return GPPD_ERR_ARG;
    }
    CK(cudaStreamSynchronize(s.stream));
    CK(cudaMemcpy(cov, s.cov.p, sizeof(double) * GPPD_COV_STRIDE * (size_t)nfits, cudaMemcpyDeviceToHost));
    return GPPD_OK;
}

int gppd_debug_harmonics(gppd_handle h, int slot, double *htab, int64_t nvals) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !htab) return GPPD_ERR_ARG;
    Slot &s = h->slots[slot];
    CK(cudaStreamSynchronize(s.stream));
    if (nvals > s.htab_vals) {
        g_last_error = "debug_harmonics: the slot's last batch has fewer values";
        return GPPD_ERR_ARG;
    }
    CK(cudaMemcpy(htab, s.htab.p, sizeof(double) * (size_t)nvals, cudaMemcpyDeviceToHost));
    return GPPD_OK;
}

int64_t gppd_launch_count(gppd_handle h) { return h ? h->launches : 0; }

int gppd_debug_counters(gppd_handle h, uint64_t *out16, int reset) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (!out16) return GPPD_ERR_ARG;
    CK(cudaDeviceSynchronize());
    tc_profile_read(reinterpret_cast<unsigned long long *>(out16), reset);
    CK(cudaGetLastError());
    return GPPD_OK;
}

int gppd_measure_fp64_peak(gppd_handle h, double *tflops) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (!tflops) return GPPD_ERR_ARG;
    Slot &s = h->slots[0];
    if ((rc = s.flags.ensure(64))) return rc;
    *tflops = measure_dfma_tflops(s.stream, s.flags.as<double>());
    h->launches += 6;
    CK(cudaGetLastError());
    return GPPD_OK;
}

int gppd_set_split_chains(gppd_handle h, int on) {
    if (!h) return GPPD_ERR_ARG;
    h->split_chains = on != 0;
    return GPPD_OK;
}

int gppd_enable_timing(gppd_handle h, int on) {
    if (!h) return GPPD_ERR_ARG;
    h->timing = on != 0;
    return GPPD_OK;
}

int gppd_pass_times(gppd_handle h, double *ms, int64_t *counts, int reset) {
    int rc = check_handle(h);
    if (rc) return rc;
    for (int p = 0; p < NPASS; ++p) {
        if (ms) ms[p] = 0.0;
        if (counts) counts[p] = 0;
    }
    for (int i = 0; i < 2 * NSLOTS; ++i) {
        PassTimer &t = (i < NSLOTS ? h->slots[i] : h->aux[i - NSLOTS]).timer;
        for (size_t k = 0; k < t.pass.size(); ++k) {
            cudaEvent_t a = t.ev[2 * k], b = t.ev[2 * k + 1];
            CK(cudaEventSynchronize(b));
            float dt = 0.f;
            CK(cudaEventElapsedTime(&dt, a, b));
            t.ms[t.pass[k]] += dt;
            t.count[t.pass[k]] += 1;
            cudaEventDestroy(a);
            cudaEventDestroy(b);
        }
        t.ev.clear();
        t.pass.clear();
        for (int p = 0; p < NPASS; ++p) {
            if (ms) ms[p] += t.ms[p];
            if (counts) counts[p] += t.count[p];
            if (reset) {
                t.ms[p] = 0.0;
                t.count[p] = 0;
            }
        }
    }
    return GPPD_OK;
}

int64_t gppd_num_windows(int64_t n, int64_t nwindow) {
    if (n <= 0) return 0;
    if (nwindow <= 0 || nwindow >= n) return 1;
    return (n + nwindow - 1) / nwindow;
}

// ---------------------------------------------------------------------------
int gppd_buildstates(gppd_handle h, int64_t n, const double *t, const double *timer1,
                     int64_t n1, const double *timer2, int64_t n2, int64_t lag,
                     double pre, double post, int8_t *state_out) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (!t || !timer1 || !timer2 || !state_out || n < 2 || n1 < 1 || n2 < 1 ||
        n1 > MAX_TIMER || n2 > MAX_TIMER) {
        g_last_error = "buildstates: need n >= 2 and non-empty timers";
        return GPPD_ERR_ARG;
    }
    Slot &s = h->slots[0];
    cudaStream_t st = s.stream;
    CK(cudaStreamSynchronize(st));
    if ((rc = s.t.ensure(sizeof(double) * (size_t)n))) return rc;
    if ((rc = s.state_out.ensure((size_t)n))) return rc;
    CK(cudaMemcpyAsync(s.t.p, t, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    std::vector<TableArgs> tabs(1);
    TableArgs &a = tabs[0];
    array_views(n, s.t.as<double>(), nullptr, nullptr, a);
    a.timer1 = timer1;
    a.timer2 = timer2;
    a.n1 = n1;
    a.n2 = n2;
    a.lag = lag;
    a.pre = pre;
    a.post = post;
    a.d_state_out = s.state_out.as<int8_t>();
    if ((rc = run_batch(h, s, st, tabs, nullptr, nullptr, true))) return rc;
    CK(cudaMemcpyAsync(state_out, s.state_out.p, (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return GPPD_OK;
}

// ---------------------------------------------------------------------------
int gppd_demodulate_f64(gppd_handle h, int64_t n, int64_t nwindow, const double *t,
                        const double *data, const int8_t *state, const gppd_options *opt,
                        double *out, double *params, double *chi2, int32_t *info,
                        double *trace) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (!t || !data || !out || !params || !chi2 || n < 2) {
        g_last_error = "demodulate_f64: null buffer or n < 2";
        return GPPD_ERR_ARG;
    }
    if ((rc = check_array_options(opt))) return rc;
    Slot &s = h->slots[0];
    cudaStream_t st = s.stream;
    CK(cudaStreamSynchronize(st));
    int64_t nwin = gppd_num_windows(n, nwindow);
    size_t nfits = (size_t)nwin * NDIODE;
    size_t cbytes = sizeof(double) * 2 * NCHAN * (size_t)n;
    if ((rc = s.t.ensure(sizeof(double) * (size_t)n))) return rc;
    if ((rc = s.data.ensure(cbytes))) return rc;
    if ((rc = s.out.ensure(cbytes))) return rc;
    if ((rc = s.params.ensure(sizeof(double) * 6 * nfits))) return rc;
    if ((rc = s.chi2.ensure(sizeof(double) * nfits))) return rc;
    if ((rc = s.info.ensure(sizeof(int) * GPPD_INFO_STRIDE * nfits))) return rc;
    if (trace)
        if ((rc = s.trace.ensure(sizeof(double) * 3 * GPPD_TRACE_MAX * nfits))) return rc;
    if (state)
        if ((rc = s.state_in.ensure((size_t)n))) return rc;
    CK(cudaMemcpyAsync(s.t.p, t, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s.data.p, data, cbytes, cudaMemcpyHostToDevice, st));
    if (state) CK(cudaMemcpyAsync(s.state_in.p, state, (size_t)n, cudaMemcpyHostToDevice, st));
    if (trace) CK(cudaMemsetAsync(s.trace.p, 0, sizeof(double) * 3 * GPPD_TRACE_MAX * nfits, st));

    std::vector<TableArgs> tabs(1);
    TableArgs &a = tabs[0];
    array_views(n, s.t.as<double>(), s.data.as<double2>(), s.out.as<double2>(), a);
    a.wrows = nwindow;
    a.d_state_in = state ? s.state_in.as<int8_t>() : nullptr;
    a.d_params = s.params.as<double>();
    a.d_chi2 = s.chi2.as<double>();
    a.d_info = s.info.as<int>();
    if ((rc = run_batch(h, s, st, tabs, opt, trace ? s.trace.as<double>() : nullptr, false)))
        return rc;

    CK(cudaMemcpyAsync(out, s.out.p, cbytes, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(params, s.params.p, sizeof(double) * 6 * nfits, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(chi2, s.chi2.p, sizeof(double) * nfits, cudaMemcpyDeviceToHost, st));
    if (info)
        CK(cudaMemcpyAsync(info, s.info.p, sizeof(int) * GPPD_INFO_STRIDE * nfits,
                           cudaMemcpyDeviceToHost, st));
    if (trace)
        CK(cudaMemcpyAsync(trace, s.trace.p, sizeof(double) * 3 * GPPD_TRACE_MAX * nfits,
                           cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return GPPD_OK;
}

int gppd_demodulate_f64_dev(gppd_handle h, int slot, void *stream, int64_t n, int64_t nwindow,
                            const double *d_t, const double *d_data, const int8_t *d_state,
                            const gppd_options *opt, double *d_out, double *d_params,
                            double *d_chi2, int32_t *d_info) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !d_t || !d_data || !d_out || !d_params || !d_chi2 || n < 2) {
        g_last_error = "demodulate_f64_dev: bad slot, null buffer or n < 2";
        return GPPD_ERR_ARG;
    }
    if ((rc = check_array_options(opt))) return rc;
    Slot &s = h->slots[slot];
    cudaStream_t st = stream ? (cudaStream_t)stream : s.stream;
    std::vector<TableArgs> tabs(1);
    TableArgs &a = tabs[0];
    array_views(n, d_t, reinterpret_cast<const double2 *>(d_data), reinterpret_cast<double2 *>(d_out), a);
    a.wrows = nwindow;
    a.d_state_in = d_state;
    a.d_params = d_params;
    a.d_chi2 = d_chi2;
    a.d_info = d_info;
    return run_batch(h, s, st, tabs, opt, nullptr, false);
}

// ---------------------------------------------------------------------------
int gppd_table_windows(int64_t n, const int32_t *time_us, double mjd, double window_s,
                       int64_t *nwindow_rows, int64_t *nwin) {
    if (!nwindow_rows || !nwin || n < 2) return GPPD_ERR_ARG;
    if (!(window_s > 0.0)) {
        *nwindow_rows = n;
        *nwin = 1;
        return GPPD_OK;
    }
    if (!time_us) return GPPD_ERR_ARG;
    // nwindow = round(Int, window / (times[2] - times[1])), ties to even,
    // reference src/GPPupilDemodulation.jl:139,192 (host code is compiled with
    // -ffp-contract=off so these are the reference's roundings)
    volatile double tmjd = 86400.0 * mjd;
    volatile double t0 = (double)time_us[0] * 1e-6;
    volatile double t1 = (double)time_us[1] * 1e-6;
    t0 = t0 + tmjd;
    t1 = t1 + tmjd;
    double w = nearbyint(window_s / (t1 - t0));
    if (!(w >= 1.0) || w > 9.0e15) {
        g_last_error = "window shorter than one row";
        return GPPD_ERR_ARG;
    }
    *nwindow_rows = (int64_t)w;
    *nwin = gppd_num_windows(n, *nwindow_rows);
    return GPPD_OK;
}

int gppd_submit_table_f32(gppd_handle h, int slot, int64_t n, const int32_t *time_us,
                          double mjd, const float *volt, const double *offsets,
                          const double *timer1, int64_t n1, const double *timer2, int64_t n2,
                          double window_s, const gppd_options *opt, float *volt_out,
                          double *params, double *chi2, int32_t *info, int8_t *state_out) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !time_us || !volt || !volt_out || !params || !chi2 || n < 2) {
        g_last_error = "process_table_f32: bad slot, null buffer or n < 2";
        return GPPD_ERR_ARG;
    }
    return stage_table(h, slot, n, time_us, volt, nullptr, false, 0, 0, 0, mjd, offsets, timer1, n1, timer2, n2,
                       window_s, opt, volt_out, params, chi2, info, state_out);
}

int gppd_submit_fits_rows(gppd_handle h, int slot, int64_t n, const void *rows, int64_t row_bytes,
                          int64_t time_off, int64_t volt_off, double mjd, const double *offsets,
                          const double *timer1, int64_t n1, const double *timer2, int64_t n2,
                          double window_s, const gppd_options *opt, void *rows_out, double *params,
                          double *chi2, int32_t *info, int8_t *state_out) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !rows || !rows_out || !params || !chi2 || n < 2) {
        g_last_error = "submit_fits_rows: bad slot, null buffer or n < 2";
        return GPPD_ERR_ARG;
    }
    return stage_table(h, slot, n, nullptr, nullptr, rows, false, row_bytes, time_off, volt_off, mjd, offsets,
                       timer1, n1, timer2, n2, window_s, opt, rows_out, params, chi2, info, state_out);
}

// ---------------------------------------------------------------------------
// native file ingest / egress (gppd_file_*)
namespace {

constexpr size_t IO_CHUNK = 8u << 20;

int io_error(const std::string &what, const std::string &path) {
    g_last_error = what + " " + path + ": " + strerror(errno);
    return GPPD_ERR_IO;
}

// reader thread: file -> pinned (chunk by chunk, each chunk uploaded while the next is read)
// -> the batch -> pinned results
int file_reader(gppd_handle h, int slot) {
    Slot &s = h->slots[slot];
    FileJob &f = s.file;
    CK(cudaSetDevice(h->device));
    int rc;
    const size_t bytes = (size_t)f.n * (size_t)f.row_bytes;
    const int out_floats = (f.opt.flags & GPPD_KEEPRAW) ? 144 : 80;
    f.row_bytes_out = f.row_bytes + 4 * (out_floats - 80);
    // worst case number of windows is not known before TIME is read: size the small result
    // buffers after the first chunk
    if ((rc = f.rows.ensure(bytes))) return rc;
    if ((rc = f.rows_out.ensure((size_t)f.n * (size_t)f.row_bytes_out))) return rc;
    if ((rc = f.state.ensure((size_t)f.n))) return rc;
    CK(cudaStreamSynchronize(s.stream));          // the slot's previous table is done with s.rows
    if ((rc = s.rows.ensure(bytes))) return rc;
    const int fd = open(f.in_path.c_str(), O_RDONLY);
    if (fd < 0) return io_error("cannot open", f.in_path);
#ifdef POSIX_FADV_SEQUENTIAL
    posix_fadvise(fd, f.data_offset, (off_t)bytes, POSIX_FADV_SEQUENTIAL);
#endif
    size_t done = 0;
    while (done < bytes) {
        const size_t want = bytes - done < IO_CHUNK ? bytes - done : IO_CHUNK;
        size_t got = 0;
        while (got < want) {
            const ssize_t r = pread(fd, f.rows.as<char>() + done + got, want - got, (off_t)(f.data_offset + done + got));
            if (r < 0 && errno == EINTR) continue;
            if (r <= 0) {
                close(fd);
                if (r == 0) errno = EIO;
                return io_error("short read of the METROLOGY records of", f.in_path);
            }
            got += (size_t)r;
        }
        cudaError_t e = cudaMemcpyAsync(s.rows.as<char>() + done, f.rows.as<char>() + done, want,
                                        cudaMemcpyHostToDevice, s.stream);
        if (e != cudaSuccess) {
            close(fd);
            g_last_error = std::string("cudaMemcpyAsync: ") + cudaGetErrorString(e);
            return GPPD_ERR_CUDA;
        }
        done += want;
    }
    close(fd);
    // number of fits (windows x 32) -> the small pinned result buffers
    int64_t wrows = f.n, nwin = 1;
    if ((rc = record_windows(f.n, f.rows.as<unsigned char>(), f.row_bytes, f.time_off, f.volt_off, f.mjd,
                             f.window_s, wrows, nwin)))
        return rc;
    f.nfits = nwin * NDIODE;
    if ((rc = f.params.ensure(sizeof(double) * 6 * (size_t)f.nfits))) return rc;
    if ((rc = f.chi2.ensure(sizeof(double) * (size_t)f.nfits))) return rc;
    if ((rc = f.info.ensure(sizeof(int32_t) * GPPD_INFO_STRIDE * (size_t)f.nfits))) return rc;
    return stage_table(h, slot, f.n, nullptr, nullptr, f.rows.p, true, f.row_bytes, f.time_off, f.volt_off, f.mjd,
                       f.have_offsets ? f.offsets : nullptr, f.faint ? f.timer1.data() : nullptr,
                       (int64_t)f.timer1.size(), f.faint ? f.timer2.data() : nullptr, (int64_t)f.timer2.size(),
                       f.window_s, &f.opt, f.rows_out.p, f.params.as<double>(), f.chi2.as<double>(),
                       f.info.as<int32_t>(), f.state.as<int8_t>());
}

int write_all(int fd, const void *buf, size_t len, const std::string &path) {
    const char *p = reinterpret_cast<const char *>(buf);
    while (len) {
        const ssize_t w = write(fd, p, len);
        if (w < 0 && errno == EINTR) continue;
        if (w <= 0) return io_error("cannot write", path);
        p += w;
        len -= (size_t)w;
    }
    return GPPD_OK;
}

struct OutSeg {
    int kind;
    int64_t offset, length;
    std::string bytes;
};

// writer thread: the output file from its segments (FITScopy!, src/FitsUtils.jl:95-156)
int file_writer(gppd_handle h, int slot, const std::string &out_path, const std::vector<OutSeg> &segs,
                const unsigned char *extra, int64_t extra_row_bytes) {
    Slot &s = h->slots[slot];
    FileJob &f = s.file;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(s.stream));          // the output records are in pinned memory
    const int fo = open(out_path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fo < 0) return io_error("cannot create", out_path);
    int fi = -1, rc = GPPD_OK;
    std::vector<char> bounce;
    for (const OutSeg &g : segs) {
        if (g.kind == GPPD_SEG_BYTES) {
            rc = write_all(fo, g.bytes.data(), g.bytes.size(), out_path);
        } else if (g.kind == GPPD_SEG_COPY) {
            if (fi < 0 && (fi = open(f.in_path.c_str(), O_RDONLY)) < 0) {
                rc = io_error("cannot open", f.in_path);
                break;
            }
            bounce.resize(IO_CHUNK);
            int64_t done = 0;
            while (done < g.length && rc == GPPD_OK) {
                const size_t want = (size_t)((g.length - done) < (int64_t)IO_CHUNK ? (g.length - done) : (int64_t)IO_CHUNK);
                const ssize_t r = pread(fi, bounce.data(), want, (off_t)(g.offset + done));
                if (r < 0 && errno == EINTR) continue;
                if (r <= 0) {
                    if (r == 0) errno = EIO;
                    rc = io_error("short read of", f.in_path);
                    break;
                }
                rc = write_all(fo, bounce.data(), (size_t)r, out_path);
                done += r;
            }
        } else if (g.kind == GPPD_SEG_RECORDS) {
            const size_t rb = (size_t)f.row_bytes_out;
            size_t total;
            if (!extra || extra_row_bytes <= 0) {
                total = (size_t)f.n * rb;
                rc = write_all(fo, f.rows_out.p, total, out_path);
            } else {    // records widened by the per-row columns of window mode
                const size_t eb = (size_t)extra_row_bytes, ob = rb + eb;
                const size_t rows_per = IO_CHUNK / ob ? IO_CHUNK / ob : 1;
                bounce.resize(rows_per * ob);
                total = (size_t)f.n * ob;
                for (int64_t r0 = 0; r0 < f.n && rc == GPPD_OK; r0 += (int64_t)rows_per) {
                    const size_t nr = (size_t)((f.n - r0) < (int64_t)rows_per ? (f.n - r0) : (int64_t)rows_per);
                    for (size_t r = 0; r < nr; ++r) {
                        memcpy(bounce.data() + r * ob, f.rows_out.as<char>() + ((size_t)r0 + r) * rb, rb);
                        memcpy(bounce.data() + r * ob + rb, extra + ((size_t)r0 + r) * eb, eb);
                    }
                    rc = write_all(fo, bounce.data(), nr * ob, out_path);
                }
            }
            const size_t pad = (2880 - total % 2880) % 2880;
            if (rc == GPPD_OK && pad) {
                const std::string zeros(pad, '\0');
                rc = write_all(fo, zeros.data(), pad, out_path);
            }
        }
        if (rc != GPPD_OK) break;
    }
    if (fi >= 0) close(fi);
    if (close(fo) != 0 && rc == GPPD_OK) rc = io_error("cannot close", out_path);
    return rc;
}

}  // namespace

int gppd_file_submit(gppd_handle h, int slot, const char *path, int64_t data_offset, int64_t n,
                     int64_t row_bytes, int64_t time_off, int64_t volt_off, double mjd,
                     const double *offsets, const double *timer1, int64_t n1,
                     const double *timer2, int64_t n2, double window_s, const gppd_options *opt) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !path || data_offset < 0 || n < 2 || row_bytes < 324 ||
        n1 < 0 || n2 < 0 || n1 > MAX_TIMER || n2 > MAX_TIMER) {
        g_last_error = "file_submit: bad slot, path, offset or table shape";
        return GPPD_ERR_ARG;
    }
    {   // I/O threads of the handle: a third of the cores read, three quarters write (measured on
        // a 16-core box, 300 files on tmpfs: 2+2 threads 1.70 s, 3+4 1.37 s, 6+12 1.15 s);
        // GPPD_IO_THREADS="readers,writers" overrides
        const int hw = (int)std::thread::hardware_concurrency();
        int nr = hw / 3 < 2 ? 2 : (hw / 3 > 6 ? 6 : hw / 3);
        int nw = hw * 3 / 4 < 3 ? 3 : (hw * 3 / 4 > 12 ? 12 : hw * 3 / 4);
        if (const char *e = getenv("GPPD_IO_THREADS")) {
            int a = 0, b = 0;
            if (sscanf(e, "%d,%d", &a, &b) == 2 && a > 0 && b > 0 && a <= 32 && b <= 32) {
                nr = a;
                nw = b;
            }
        }
        h->readers.start(nr, h->device);
        h->writers.start(nw, h->device);
    }
    FileJob &f = h->slots[slot].file;
    {
        std::unique_lock<std::mutex> lk(f.m);
        f.cv.wait(lk, [&f] { return !(f.stage == 1 || f.stage == 3 || f.write_pending); });
        f.stage = 1;
        f.rc = GPPD_OK;
        f.err.clear();
        f.in_path = path;
        f.data_offset = data_offset;
        f.n = n;
        f.row_bytes = row_bytes;
        f.time_off = time_off;
        f.volt_off = volt_off;
        f.mjd = mjd;
        f.window_s = window_s;
        f.have_offsets = offsets != nullptr;
        if (offsets) memcpy(f.offsets, offsets, sizeof f.offsets);
        f.faint = timer1 && timer2 && n1 > 0 && n2 > 0;
        f.timer1.assign(f.faint ? timer1 : nullptr, f.faint ? timer1 + n1 : nullptr);
        f.timer2.assign(f.faint ? timer2 : nullptr, f.faint ? timer2 + n2 : nullptr);
        memset(&f.opt, 0, sizeof f.opt);
        if (opt) f.opt = *opt;
    }
    h->readers.post([h, slot] {
        FileJob &f = h->slots[slot].file;
        const int r = file_reader(h, slot);
        std::lock_guard<std::mutex> lk(f.m);
        f.rc = r;
        if (r) f.err = g_last_error;
        f.stage = 2;
        f.cv.notify_all();
    });
    return GPPD_OK;
}

int gppd_file_wait(gppd_handle h, int slot, double *params, double *chi2, int32_t *info,
                   int8_t *state_out) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS) return GPPD_ERR_ARG;
    Slot &s = h->slots[slot];
    FileJob &f = s.file;
    {
        std::unique_lock<std::mutex> lk(f.m);
        if (f.stage == 0) {
            g_last_error = "file_wait: no file was submitted on this slot";
            return GPPD_ERR_ARG;
        }
        f.cv.wait(lk, [&f] { return f.stage != 1; });
        if (f.rc) {
            g_last_error = f.err;
            return f.rc;
        }
    }
    CK(cudaStreamSynchronize(s.stream));
    if (params) memcpy(params, f.params.p, sizeof(double) * 6 * (size_t)f.nfits);
    if (chi2) memcpy(chi2, f.chi2.p, sizeof(double) * (size_t)f.nfits);
    if (info) memcpy(info, f.info.p, sizeof(int32_t) * GPPD_INFO_STRIDE * (size_t)f.nfits);
    if (state_out && f.faint) memcpy(state_out, f.state.p, (size_t)f.n);
    return GPPD_OK;
}

int gppd_file_write(gppd_handle h, int slot, const char *out_path, const gppd_file_segment *segs,
                    int32_t nsegs, const void *extra, int64_t extra_row_bytes) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || !out_path || !segs || nsegs < 1 || (extra && extra_row_bytes <= 0)) {
        g_last_error = "file_write: bad slot, path or segments";
        return GPPD_ERR_ARG;
    }
    FileJob &f = h->slots[slot].file;
    std::vector<OutSeg> copy((size_t)nsegs);
    for (int i = 0; i < nsegs; ++i) {
        copy[i].kind = segs[i].kind;
        copy[i].offset = segs[i].offset;
        copy[i].length = segs[i].length;
        if (segs[i].kind == GPPD_SEG_BYTES) {
            if (!segs[i].bytes || segs[i].length < 0) return GPPD_ERR_ARG;
            copy[i].bytes.assign(reinterpret_cast<const char *>(segs[i].bytes), (size_t)segs[i].length);
        } else if (segs[i].kind != GPPD_SEG_COPY && segs[i].kind != GPPD_SEG_RECORDS) {
            g_last_error = "file_write: unknown segment kind";
            return GPPD_ERR_ARG;
        }
    }
    {
        std::lock_guard<std::mutex> lk(f.m);
        if (f.stage == 0 || f.stage == 3 || f.write_pending) {
            g_last_error = "file_write: no file waiting to be written on this slot";
            return GPPD_ERR_ARG;
        }
        f.write_pending = true;
    }
    const std::string out(out_path);
    const unsigned char *ex = reinterpret_cast<const unsigned char *>(extra);
    h->writers.post([h, slot, out, copy, ex, extra_row_bytes] {
        FileJob &f = h->slots[slot].file;
        {
            std::unique_lock<std::mutex> lk(f.m);
            f.cv.wait(lk, [&f] { return f.stage == 2; });
            f.stage = 3;
        }
        int r = f.rc;       // a failed read / fit: nothing to write
        std::string e = f.err;
        if (r == GPPD_OK) {
            r = file_writer(h, slot, out, copy, ex, extra_row_bytes);
            if (r) e = g_last_error;
        }
        std::lock_guard<std::mutex> lk(f.m);
        f.rc = r;
        f.err = e;
        f.stage = 0;
        f.write_pending = false;
        f.cv.notify_all();
    });
    return GPPD_OK;
}

int gppd_file_drain(gppd_handle h) {
    int rc = check_handle(h);
    if (rc) return rc;
    int first = GPPD_OK;
    for (int i = 0; i < NSLOTS; ++i) {
        FileJob &f = h->slots[i].file;
        std::unique_lock<std::mutex> lk(f.m);
        f.cv.wait(lk, [&f] { return !(f.stage == 1 || f.stage == 3 || f.write_pending); });
        if (f.rc && first == GPPD_OK) {
            first = f.rc;
            g_last_error = f.err;
        }
        f.rc = GPPD_OK;
    }
    return first;
}

int gppd_wait(gppd_handle h, int slot) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS) return GPPD_ERR_ARG;
    CK(cudaStreamSynchronize(h->slots[slot].stream));
    return GPPD_OK;
}

int gppd_process_table_f32(gppd_handle h, int64_t n, const int32_t *time_us, double mjd,
                           const float *volt, const double *offsets, const double *timer1,
                           int64_t n1, const double *timer2, int64_t n2, double window_s,
                           const gppd_options *opt, float *volt_out, double *params,
                           double *chi2, int32_t *info, int8_t *state_out) {
    int rc = gppd_submit_table_f32(h, 0, n, time_us, mjd, volt, offsets, timer1, n1, timer2, n2,
                                   window_s, opt, volt_out, params, chi2, info, state_out);
    if (rc) return rc;
    return gppd_wait(h, 0);
}

int gppd_process_tables_f32_dev(gppd_handle h, int slot, void *stream, int64_t ntables,
                                const int64_t *n, const int64_t *nwindow_rows,
                                const int32_t *const *d_time_us, const double *mjd,
                                const float *const *d_volt, const double *d_offsets,
                                const double *const *timer1, const int64_t *n1,
                                const double *const *timer2, const int64_t *n2,
                                const gppd_options *opt, float *const *d_volt_out,
                                double *const *d_params, double *const *d_chi2,
                                int32_t *const *d_info, int8_t *const *d_state_out) {
    int rc = check_handle(h);
    if (rc) return rc;
    if (slot < 0 || slot >= NSLOTS || ntables < 1 || !n || !d_time_us || !mjd || !d_volt ||
        !d_volt_out || !d_params || !d_chi2) {
        g_last_error = "process_tables_f32_dev: bad slot or null array";
        return GPPD_ERR_ARG;
    }
    for (int64_t t = 0; t < ntables; ++t) {
        if (!d_time_us[t] || !d_volt[t] || !d_volt_out[t] || !d_params[t] || !d_chi2[t] || n[t] < 2) {
            g_last_error = "process_tables_f32_dev: null table buffer or n < 2";
            return GPPD_ERR_ARG;
        }
    }
    gppd_options o;
    if ((rc = table_options(opt, d_offsets != nullptr, o))) return rc;
    std::vector<TableArgs> tabs((size_t)ntables);
    for (int64_t t = 0; t < ntables; ++t) {
        TableArgs &a = tabs[(size_t)t];
        table_views(n[t], mjd[t], d_time_us[t], d_volt[t], d_offsets, d_volt_out[t], o.flags, a);
        a.wrows = nwindow_rows ? nwindow_rows[t] : 0;
        const bool faint = timer1 && timer2 && n1 && n2 && timer1[t] && timer2[t] && n1[t] > 0 &&
                           n2[t] > 0;
        a.timer1 = faint ? timer1[t] : nullptr;
        a.timer2 = faint ? timer2[t] : nullptr;
        a.n1 = faint ? n1[t] : 0;
        a.n2 = faint ? n2[t] : 0;
        a.d_params = d_params[t];
        a.d_chi2 = d_chi2[t];
        a.d_info = d_info ? d_info[t] : nullptr;
        a.d_state_out = d_state_out ? d_state_out[t] : nullptr;
    }
    return run_tables(h, slot, stream ? (cudaStream_t)stream : h->slots[slot].stream, tabs, o);
}

int gppd_process_table_f32_dev(gppd_handle h, int slot, void *stream, int64_t n,
                               int64_t nwindow_rows, const int32_t *d_time_us, double mjd,
                               const float *d_volt, const double *d_offsets,
                               const double *timer1, int64_t n1, const double *timer2,
                               int64_t n2, const gppd_options *opt, float *d_volt_out,
                               double *d_params, double *d_chi2, int32_t *d_info,
                               int8_t *d_state_out) {
    return gppd_process_tables_f32_dev(h, slot, stream, 1, &n, &nwindow_rows, &d_time_us, &mjd,
                                       &d_volt, d_offsets, &timer1, &n1, &timer2, &n2, opt,
                                       &d_volt_out, &d_params, &d_chi2, d_info ? &d_info : nullptr,
                                       d_state_out ? &d_state_out : nullptr);
}

}  // extern "C"
