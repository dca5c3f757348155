// stream_kernels.cu -- the HBM-bound passes around the fit, batched over the
// tables of one launch sequence (blockIdx.y selects the table or the job group):
//   * FAINT segmentation (reference buildstates, src/Faint.jl:21-73)
//   * per-row sin/cos basis of theta = fl(omega t) and per-job theta range
//   * per-state mean/variance of |d| (reference compute_mean_var_power,
//     src/Faint.jl:89-100), two partial-sum passes like the reference's two passes
//   * demodulation + repack (reference src/Modulation.jl:417-425 and
//     src/GPPupilDemodulation.jl:163-171,253)
#include "fit_math.cuh"
#include "gppd_device.cuh"
#include "kernels.h"
#include "tma.cuh"

namespace gppd {

// ---------------------------------------------------------------------------
// order-preserving map double -> uint64 for atomicMin/atomicMax
__device__ __forceinline__ unsigned long long f64_key(double x) {
    unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double f64_unkey(unsigned long long k) {
    unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// ===========================================================================
// Segmentation.  The reference scans the rows serially carrying two timer
// queues; at most one event per queue fires per row.  With non-decreasing
// timestamps the row at which the k-th event of a queue fires is
//     trig_k = max(trig_{k-1} + 1, lower_bound(t, event_k))
// so the scan reduces to (1) lower bounds of all timer values (parallel),
// (2) a serial merge over the O(100) events, (3) a parallel fill.
// Non-monotonic timestamps take the serial path, statement for statement.
// ===========================================================================
struct SegEvent {
    long long row;
    long long forget;
    int state;
    int pad;
};
static_assert(sizeof(SegEvent) == SEG_EVENT_BYTES, "SegEvent size");

__global__ void k_seg_init(const TableDesc *tabs) {
    const TableDesc &tb = tabs[blockIdx.x];
    if (tb.seg.n1 > 0 && threadIdx.x < 2) tb.seg.flags[threadIdx.x] = 0;
}

__global__ void k_seg_monotone(const TableDesc *tabs) {
    const TableDesc &tb = tabs[blockIdx.y];
    if (tb.seg.n1 <= 0) return;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    bool bad = false;
    for (; i + 1 < tb.tv.n; i += stride) {
        double a = row_time(tb.tv, i), b = row_time(tb.tv, i + 1);
        if (!(b >= a)) bad = true;
    }
    if (bad) tb.seg.flags[1] = 1;
}

__device__ long long seg_lower_bound(const TableView &tv, double v) {
    long long lo = 0, hi = tv.n;  // first i with t[i] >= v
    while (lo < hi) {
        long long mid = (lo + hi) >> 1;
        if (row_time(tv, mid) >= v) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__global__ void k_seg_lower_bounds(const TableDesc *tabs) {
    const TableDesc &tb = tabs[blockIdx.y];
    const SegDesc &sp = tb.seg;
    if (sp.n1 <= 0) return;
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    int tot = sp.n1 + 1 + sp.n2 + 1;
    if (k >= tot) return;
    double timestep = row_time(tb.tv, 1) - row_time(tb.tv, 0);   // src/Faint.jl:24
    double shift = (double)sp.lag * timestep;                    // :25-26
    double tlast = row_time(tb.tv, tb.tv.n - 1);
    long long *lb1 = sp.lb, *lb2 = sp.lb + (sp.n1 + 1);
    if (k <= sp.n1) {
        double v = (k < sp.n1) ? __dadd_rn(sp.timer1[k], shift) : tlast;
        lb1[k] = seg_lower_bound(tb.tv, v);
    } else {
        int j = k - sp.n1 - 1;
        double v = (j < sp.n2) ? __dadd_rn(sp.timer2[j], shift) : tlast;
        lb2[j] = seg_lower_bound(tb.tv, v);
    }
}

__device__ __forceinline__ long long seg_ceil_count(double delay, double timestep) {
    double r = ceil(delay / timestep);                           // :29-30
    if (!(r > 0.0)) return 0;
    if (r > 4.0e18) return 4000000000000000000ll;
    return (long long)r;
}

// serial merge of the two event queues (one thread per table)
__global__ void k_seg_events(const TableDesc *tabs) {
    if (threadIdx.x != 0) return;
    const TableDesc &tb = tabs[blockIdx.x];
    const SegDesc &sp = tb.seg;
    if (sp.n1 <= 0 || sp.flags[1]) return;  // bright, or non-monotone: serial path
    const TableView &tv = tb.tv;
    SegEvent *events = reinterpret_cast<SegEvent *>(sp.events);
    const long long *lb1 = sp.lb, *lb2 = sp.lb + (sp.n1 + 1);
    double timestep = row_time(tv, 1) - row_time(tv, 0);
    double shift = (double)sp.lag * timestep;
    double tlast = row_time(tv, tv.n - 1);
    long long premax = seg_ceil_count(sp.pre, timestep);
    long long postmax = seg_ceil_count(sp.post, timestep);
    long long lb_last = lb1[sp.n1];
    int i1 = 0, i2 = 0;                       // next queue element to pop
    double first1 = __dadd_rn(sp.timer1[i1], shift); long long lbh1 = lb1[i1]; ++i1;
    double first2 = __dadd_rn(sp.timer2[i2], shift); long long lbh2 = lb2[i2]; ++i2;
    long long last1 = -1, last2 = -1;
    int cur = ST_NORMAL;
    int ne = 0;
    for (;;) {
        long long tr1 = lbh1 > last1 + 1 ? lbh1 : last1 + 1;
        long long tr2 = lbh2 > last2 + 1 ? lbh2 : last2 + 1;
        long long row = tr1 < tr2 ? tr1 : tr2;
        if (row >= tv.n) break;
        long long forget = 0;
        bool fired = false;
        if (tr1 == row) {                      // :40-52
            cur = ST_HIGH;
            forget = premax;
            fired = true;
            if (i1 >= sp.n1) {
                first1 = tlast; lbh1 = lb_last;
                if (first2 == tlast) cur = ST_NORMAL;
            } else {
                first1 = __dadd_rn(sp.timer1[i1], shift); lbh1 = lb1[i1]; ++i1;
            }
            last1 = row;
        }
        if (tr2 == row) {                      // :54-65
            cur = ST_LOW;
            forget = postmax;
            fired = true;
            if (i2 >= sp.n2) {
                first2 = tlast; lbh2 = lb_last;
                if (first1 == tlast) cur = ST_NORMAL;
            } else {
                first2 = __dadd_rn(sp.timer2[i2], shift); lbh2 = lb2[i2]; ++i2;
            }
            last2 = row;
        }
        if (fired) {
            if (ne >= sp.max_events) { sp.flags[1] = 1; return; }
            SegEvent ev; ev.row = row; ev.forget = forget; ev.state = cur; ev.pad = 0;
            events[ne++] = ev;
        }
    }
    sp.flags[0] = ne;
}

__global__ void k_seg_fill(const TableDesc *tabs) {
    const TableDesc &tb = tabs[blockIdx.y];
    const SegDesc &sp = tb.seg;
    if (sp.n1 <= 0 || sp.flags[1]) return;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= tb.tv.n) return;
    const SegEvent *events = reinterpret_cast<const SegEvent *>(sp.events);
    int ne = sp.flags[0];
    int lo = 0, hi = ne;  // last event with row <= i
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (events[mid].row <= i) lo = mid + 1; else hi = mid;
    }
    int st = ST_NORMAL;
    if (lo > 0) {
        SegEvent ev = events[lo - 1];
        st = (i - ev.row < ev.forget) ? ST_TRANSIENT : ev.state;   // :66-71
    }
    tb.state[i] = (int8_t)st;
}

// the reference's loop, statement for statement (fallback, one thread per table)
__global__ void k_seg_serial(const TableDesc *tabs) {
    if (threadIdx.x != 0) return;
    const TableDesc &tb = tabs[blockIdx.x];
    const SegDesc &sp = tb.seg;
    if (sp.n1 <= 0 || !sp.flags[1]) return;
    const TableView &tv = tb.tv;
    double timestep = row_time(tv, 1) - row_time(tv, 0);
    double shift = (double)sp.lag * timestep;
    double tlast = row_time(tv, tv.n - 1);
    long long premax = seg_ceil_count(sp.pre, timestep);
    long long postmax = seg_ceil_count(sp.post, timestep);
    int i1 = 0, i2 = 0;
    double first1 = __dadd_rn(sp.timer1[i1++], shift);
    double first2 = __dadd_rn(sp.timer2[i2++], shift);
    int cur = ST_NORMAL;
    long long forget = 0;
    for (long long k = 0; k < tv.n; ++k) {
        double time = row_time(tv, k);
        if (time >= first1) {
            cur = ST_HIGH; forget = premax;
            if (i1 >= sp.n1) { first1 = tlast; if (first2 == tlast) cur = ST_NORMAL; }
            else first1 = __dadd_rn(sp.timer1[i1++], shift);
        }
        if (time >= first2) {
            cur = ST_LOW; forget = postmax;
            if (i2 >= sp.n2) { first2 = tlast; if (first1 == tlast) cur = ST_NORMAL; }
            else first2 = __dadd_rn(sp.timer2[i2++], shift);
        }
        if (forget > 0) { tb.state[k] = (int8_t)ST_TRANSIENT; --forget; }
        else tb.state[k] = (int8_t)cur;
    }
}

void launch_segmentation(const Launcher &L, const TableDesc *d_tabs, int ntables,
                         long long max_rows, int max_timers) {
    int rb = (int)((max_rows + 255) / 256);
    int mono = rb > 296 ? 296 : rb;
    k_seg_init<<<ntables, 32, 0, L.stream>>>(d_tabs);
    k_seg_monotone<<<dim3(mono, ntables), 256, 0, L.stream>>>(d_tabs);
    k_seg_lower_bounds<<<dim3((max_timers + 2 + 127) / 128, ntables), 128, 0, L.stream>>>(d_tabs);
    k_seg_events<<<ntables, 32, 0, L.stream>>>(d_tabs);
    k_seg_fill<<<dim3(rb, ntables), 256, 0, L.stream>>>(d_tabs);
    k_seg_serial<<<ntables, 32, 0, L.stream>>>(d_tabs);
    *L.counter += 6;
}

// ===========================================================================
// Basis: (sin theta, cos theta) per row with full-accuracy reduction of the
// ~3e10 rad argument, done ONCE per row instead of once per objective call,
// plus the per-job theta range and valid-row count.
// ===========================================================================
// per-job counters: [0] valid rows, [1 + s] first row (within the job) of state s
constexpr int JOBCNT = 5;

__global__ void k_init_thkeys(unsigned long long *thkeys, int *nvalid, int njobs) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= njobs) return;
    thkeys[2 * j] = ~0ull;
    thkeys[2 * j + 1] = 0ull;
    nvalid[JOBCNT * j] = 0;
    for (int s = 0; s < 4; ++s) nvalid[JOBCNT * j + 1 + s] = 0x7fffffff;
}

constexpr int BASIS_RPT = 4;          // rows per thread, 1024 per block

__global__ void __launch_bounds__(256) k_basis(const TableDesc *tabs, unsigned flags,
                                               unsigned long long *thkeys, int *nvalid) {
    __shared__ unsigned long long s_min[8], s_max[8];
    __shared__ int s_cnt[8];
    const TableDesc &tbg = tabs[blockIdx.y];
    // table description in registers (one round trip instead of one per use)
    const TableView tv = tbg.tv;
    const long long n = tv.n, wrows = tbg.wrows;
    const int job0 = tbg.job0, njobs = tbg.njobs;
    const int8_t *state = tbg.state;
    double2 *basis = tbg.basis;
    const long long base = (long long)blockIdx.x * (256 * BASIS_RPT);
    if (base >= n) return;
    // the theta of the thread's rows first (independent loads), then the arithmetic
    double th[BASIS_RPT];
#pragma unroll
    for (int j = 0; j < BASIS_RPT; ++j) {
        const long long i = base + j * 256 + threadIdx.x;
        th[j] = i < n ? row_theta(tv, i) : 0.0;
    }
    const long long last = (base + 256 * BASIS_RPT < n ? base + 256 * BASIS_RPT : n) - 1;
    const long long jfirst = njobs == 1 ? 0 : base / wrows, jlast = njobs == 1 ? 0 : last / wrows;
    const bool one_job = jfirst == jlast;          // block-uniform
    unsigned long long kmin = ~0ull, kmax = 0ull;
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < BASIS_RPT; ++j) {
        const long long i = base + j * 256 + threadIdx.x;
        if (i >= n) continue;
        double s, c;
        sincos_large(th[j], &s, &c);
        basis[i] = make_double2(s, c);
        const long long jl = one_job ? jfirst : i / wrows;
        const unsigned long long key = f64_key(th[j]);
        int valid = 1;
        if (state) {
            const int st = state[i];
            valid = row_valid(st, flags) ? 1 : 0;
            // first row of every run of a state: candidates for the job's first row of it
            const long long il = i - jl * wrows;
            if (valid && st >= 0 && st <= 3 && (il == 0 || state[i - 1] != st))
                atomicMin(nvalid + JOBCNT * (job0 + jl) + 1 + st, (int)il);
        }
        if (one_job) {
            kmin = key < kmin ? key : kmin;
            kmax = key > kmax ? key : kmax;
            cnt += valid;
        } else {      // a block straddling jobs (small windows): per-row atomics
            atomicMin(thkeys + 2 * (job0 + jl), key);
            atomicMax(thkeys + 2 * (job0 + jl) + 1, key);
            if (valid) atomicAdd(nvalid + JOBCNT * (job0 + jl), 1);
        }
    }
    if (!one_job) return;
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long a = __shfl_xor_sync(0xffffffffu, kmin, o);
        const unsigned long long b = __shfl_xor_sync(0xffffffffu, kmax, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        kmin = a < kmin ? a : kmin;
        kmax = b > kmax ? b : kmax;
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { s_min[w] = kmin; s_max[w] = kmax; s_cnt[w] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; ++k) {
            kmin = s_min[k] < kmin ? s_min[k] : kmin;
            kmax = s_max[k] > kmax ? s_max[k] : kmax;
            cnt += s_cnt[k];
        }
        const long long job = job0 + jfirst;
        atomicMin(thkeys + 2 * job, kmin);
        atomicMax(thkeys + 2 * job + 1, kmax);
        if (cnt) atomicAdd(nvalid + JOBCNT * job, cnt);
    }
}

__global__ void k_jobinfo(const TableDesc *tabs, const unsigned long long *thkeys,
                          const int *nvalid, JobInfo *jobs) {
    int t = blockIdx.y;
    const TableDesc &tb = tabs[t];
    int jl = blockIdx.x * blockDim.x + threadIdx.x;
    if (jl >= tb.njobs) return;
    int j = tb.job0 + jl;
    JobInfo ji;
    ji.thmin = f64_unkey(thkeys[2 * j]);
    ji.thmax = f64_unkey(thkeys[2 * j + 1]);
    ji.row0 = (long long)jl * tb.wrows;
    long long rem = tb.tv.n - ji.row0;
    ji.nrows = (int)(rem < tb.wrows ? rem : tb.wrows);
    ji.nvalid = nvalid[JOBCNT * j];
    ji.table = t;
    ji.pad = 0;
    jobs[j] = ji;
}

void launch_basis(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                  int max_jobs_per_table, int njobs, unsigned flags,
                  unsigned long long *d_thkeys, int *d_nvalid, JobInfo *d_jobs) {
    k_init_thkeys<<<(njobs + 255) / 256, 256, 0, L.stream>>>(d_thkeys, d_nvalid, njobs);
    k_basis<<<dim3((unsigned)((max_rows + 256 * BASIS_RPT - 1) / (256 * BASIS_RPT)), ntables), 256, 0, L.stream>>>(
        d_tabs, flags, d_thkeys, d_nvalid);
    k_jobinfo<<<dim3((max_jobs_per_table + 127) / 128, ntables), 128, 0, L.stream>>>(
        d_tabs, d_thkeys, d_nvalid, d_jobs);
    *L.counter += 3;
}

// ===========================================================================
// Per-state statistics of |d| (FAINT; reference compute_mean_var_power,
// src/Faint.jl:89-100: mean(|d|) and 1 / var(|d|; mean) per state over the valid
// rows).  ONE streaming pass: per (diode, state) the sums of (x - p) and (x - p)^2,
// x = |d|, around a pivot p = |d| at the job's first row of that state (found by the
// basis pass), so that  mean = p + S1/n,  sum (x - mean)^2 = S2 - S1^2/n  without the
// cancellation of raw moments.  One block per (job, group, FIXED segment of
// STATS_SEG_ROWS rows); k_stats_final adds the segments of a job in index order.
// ===========================================================================
// |d| of one sample (sqrt() is correctly rounded; an rsqrt-based form measured slower)
__device__ __forceinline__ double abs_fast(double2 d) { return sqrt(fma(d.x, d.x, d.y * d.y)); }

constexpr int STATS_THREADS = 256;                          // 32 rows x 8 groups per iteration
constexpr int STATS_ITERS = STATS_SEG_ROWS / 32;            // iterations per segment
constexpr int STATS_BATCH = 4;                              // rows loaded ahead of their use

// One block per (job, segment) for all 8 groups; thread (row lane, group) like the
// demod pass, so that a warp reads 4 rows x 256 contiguous bytes.  States come in runs
// of hundreds of rows: a thread keeps the sums of ONE state in registers (9 doubles)
// and folds them into the warp's shared-memory totals when the warp's state changes
// (32-row groups that straddle a run boundary take the states one after the other).
__global__ void __launch_bounds__(STATS_THREADS, 2)
k_stats_seg(const TableDesc *tabs, const JobInfo *jobs, const int *faint_jobs, const int *jobcnt,
            unsigned flags, int P, double *part) {
    __shared__ double s_piv[NGROUP][16];
    __shared__ double s_acc[STATS_THREADS / 32][NGROUP][STATS_VALS];
    // 1-D grid, block = (FAINT job, segment): a 1e8-row job has more segments than
    // gridDim.y holds
    const int p = (int)(blockIdx.x % (unsigned)P);
    const int job = faint_jobs[blockIdx.x / (unsigned)P];
    const JobInfo ji = jobs[job];
    const TableDesc &tb = tabs[ji.table];
    if (!tb.state) return;
    const long long seg0 = (long long)p * STATS_SEG_ROWS;
    if (seg0 >= ji.nrows) return;
    const int nseg = (int)((ji.nrows - seg0) < STATS_SEG_ROWS ? (ji.nrows - seg0) : STATS_SEG_ROWS);
    const TableView tv = tb.tv;
    const int8_t *state = tb.state;
    const bool vec = tv.kind == 0 && !tv.big_endian && (tv.volt_stride & 15) == 0 &&
                     (reinterpret_cast<unsigned long long>(tv.volt) & 15ull) == 0;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rl = threadIdx.x >> 3, group = threadIdx.x & 7;
    if (threadIdx.x < 128) {   // pivots: |d| at the job's first row of each state
        const int g = threadIdx.x >> 4, dio = (threadIdx.x >> 2) & 3, st = threadIdx.x & 3;
        const int first = jobcnt[JOBCNT * job + 1 + st];
        double pv = 0.0;
        if (first != 0x7fffffff) {
            pv = abs_fast(row_sample(tv, ji.row0 + first, g * 4 + dio));
        }
        s_piv[g][dio * 4 + st] = pv;
    }
    for (int k = threadIdx.x; k < (STATS_THREADS / 32) * NGROUP * STATS_VALS; k += STATS_THREADS)
        (&s_acc[0][0][0])[k] = 0.0;
    double2 off[4];
#pragma unroll
    for (int d = 0; d < 4; ++d)
        off[d] = (tv.kind == 0 && tv.offsets) ? __ldg(tv.offsets + group * 4 + d) : make_double2(0.0, 0.0);
    __syncthreads();

    int cur = -1;                 // state whose sums the registers hold (warp-uniform)
    double a1[4], a2[4], ac = 0.0;
#pragma unroll
    for (int d = 0; d < 4; ++d) a1[d] = a2[d] = 0.0;
    // registers -> the warp's shared totals: [0..3] counts, [4..19] S1, [20..35] S2 per group;
    // the 4 rows a warp holds per group are lanes g, g + 8, g + 16, g + 24
    auto flush = [&]() {
        if (cur < 0) return;
        double v[9] = {ac, a1[0], a1[1], a1[2], a1[3], a2[0], a2[1], a2[2], a2[3]};
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            v[k] += __shfl_xor_sync(0xffffffffu, v[k], 8);
            v[k] += __shfl_xor_sync(0xffffffffu, v[k], 16);
        }
        if (lane < NGROUP) {
            double *acc = s_acc[w][lane];
            acc[cur] += v[0];
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                acc[4 + d * 4 + cur] += v[1 + d];
                acc[20 + d * 4 + cur] += v[5 + d];
            }
        }
        ac = 0.0;
#pragma unroll
        for (int d = 0; d < 4; ++d) a1[d] = a2[d] = 0.0;
    };

#pragma unroll 1
    for (int j0 = 0; j0 < STATS_ITERS; j0 += STATS_BATCH) {
        float4 ra[STATS_BATCH], rb[STATS_BATCH];
        int rs[STATS_BATCH];
#pragma unroll
        for (int j = 0; j < STATS_BATCH; ++j) {
            const int i = (j0 + j) * 32 + rl;
            rs[j] = -1;
            if (i < nseg) {
                const long long r = ji.row0 + seg0 + i;
                if (vec) {
                    const float4 *q = reinterpret_cast<const float4 *>(
                        reinterpret_cast<const char *>(tv.volt) + r * tv.volt_stride + 32 * group);
                    ra[j] = __ldg(q);
                    rb[j] = __ldg(q + 1);
                }
                const int st = state[r];
                rs[j] = (row_valid(st, flags) && st >= 0 && st <= 3) ? st : -1;
            }
        }
#pragma unroll
        for (int j = 0; j < STATS_BATCH; ++j) {
            const int i = (j0 + j) * 32 + rl;
            const int st = rs[j];
            double x[4] = {0.0, 0.0, 0.0, 0.0};
            if (st >= 0) {
                double2 dd[4];
                if (vec) {
                    dd[0] = make_double2((double)ra[j].x - off[0].x, (double)ra[j].y - off[0].y);
                    dd[1] = make_double2((double)ra[j].z - off[1].x, (double)ra[j].w - off[1].y);
                    dd[2] = make_double2((double)rb[j].x - off[2].x, (double)rb[j].y - off[2].y);
                    dd[3] = make_double2((double)rb[j].z - off[3].x, (double)rb[j].w - off[3].y);
                } else {
                    const long long r = ji.row0 + seg0 + i;
#pragma unroll
                    for (int dio = 0; dio < 4; ++dio) dd[dio] = row_sample(tv, r, group * 4 + dio);
                }
#pragma unroll
                for (int dio = 0; dio < 4; ++dio)
                    x[dio] = abs_fast(dd[dio]) - s_piv[group][dio * 4 + st];
            }
            const int st0 = __shfl_sync(0xffffffffu, st, 0);
            if (__all_sync(0xffffffffu, st == st0)) {        // the usual case: one state (or no valid row)
                if (st0 >= 0) {
                    if (st0 != cur) { flush(); cur = st0; }
                    ac += 1.0;
#pragma unroll
                    for (int dio = 0; dio < 4; ++dio) {
                        a1[dio] += x[dio];
                        a2[dio] = fma(x[dio], x[dio], a2[dio]);
                    }
                }
            } else {                                          // a run boundary inside the warp's 4 rows
#pragma unroll 1
                for (int s = 0; s < 4; ++s) {
                    if (!__any_sync(0xffffffffu, st == s)) continue;
                    if (s != cur) { flush(); cur = s; }
                    if (st == s) {
                        ac += 1.0;
#pragma unroll
                        for (int dio = 0; dio < 4; ++dio) {
                            a1[dio] += x[dio];
                            a2[dio] = fma(x[dio], x[dio], a2[dio]);
                        }
                    }
                }
            }
        }
    }
    flush();
    __syncthreads();
    for (int k = threadIdx.x; k < NGROUP * STATS_VALS; k += STATS_THREADS) {
        const int g = k / STATS_VALS, v = k - g * STATS_VALS;
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < STATS_THREADS / 32; ++j) sum += s_acc[j][g][v];
        part[((long long)(job * NGROUP + g) * P + p) * STATS_VALS + v] = sum;
    }
}

// The same sums for dense tables (rows of 80 floats back to back, 16-byte aligned: every table
// that comes through the table entry points): every WARP streams its own 128 consecutive
// rows of the segment through a private ring of cp.async.bulk stages (4 rows each, own
// mbarriers, no block-level barrier in the loop), like k_demod.  The loads of the next three
// stages are in flight while a stage is reduced, and no register holds data that is not
// being used: k_stats_seg spends 128 registers on a load batch that it cannot overlap with
// its arithmetic (ncu: long_scoreboard the top stall, 16 warps per SM); this one fits three
// blocks = 24 warps per SM.  The states of 32 rows are read one per lane, 32 rows ahead.  Thread = (row of the stage's half, group).
#ifndef ST_MT_N
#define ST_MT_N 4
#endif
#ifndef ST_MINB
#define ST_MINB 3
#endif
constexpr int ST_MT = ST_MT_N;                              // rows per stage (4 or 8)
constexpr int ST_WROWS = STATS_SEG_ROWS / (STATS_THREADS / 32);   // 128 rows per warp
constexpr int ST_STAGES = 4;
constexpr int ST_STAGE_BYTES = ST_MT * 320;
constexpr int ST_WARP_BYTES = ST_STAGES * ST_STAGE_BYTES;
constexpr int ST_SMEM = (STATS_THREADS / 32) * ST_WARP_BYTES;
constexpr int ST_PER32 = 32 / ST_MT;                        // stages per 32 rows (one state prefetch)
static_assert(ST_WROWS % 32 == 0 && (ST_MT == 4 || ST_MT == 8), "the state prefetch covers 32 rows");

template <bool BE>
__global__ void __launch_bounds__(STATS_THREADS, ST_MINB)
k_stats_seg_bulk(const TableDesc *tabs, const JobInfo *jobs, const int *faint_jobs, const int *jobcnt,
                 unsigned flags, int P, double *part) {
    extern __shared__ __align__(128) unsigned char st_smem[];
    __shared__ uint64_t s_bars[STATS_THREADS / 32][ST_STAGES];
    __shared__ double s_piv[16][NGROUP];
    __shared__ double s_acc[STATS_THREADS / 32][NGROUP][STATS_VALS];
    const int p = (int)(blockIdx.x % (unsigned)P);
    const int job = faint_jobs[blockIdx.x / (unsigned)P];
    const JobInfo ji = jobs[job];
    const TableDesc &tb = tabs[ji.table];
    if (!tb.state) return;
    const long long seg0 = (long long)p * STATS_SEG_ROWS;
    if (seg0 >= ji.nrows) return;
    const int nseg = (int)((ji.nrows - seg0) < STATS_SEG_ROWS ? (ji.nrows - seg0) : STATS_SEG_ROWS);
    const TableView tv = tb.tv;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rl = lane >> 3, group = lane & 7;

    // this warp's rows and the first loads, before anything else
    const int wr0 = w * ST_WROWS;
    const int wn = nseg - wr0 < ST_WROWS ? nseg - wr0 : ST_WROWS;          // may be <= 0
    const int nmt = wn > 0 ? (wn + ST_MT - 1) / ST_MT : 0;
    const long long row0 = ji.row0 + seg0 + wr0;                           // table row of the warp's first row
    unsigned char *ring = st_smem + w * ST_WARP_BYTES;
    uint64_t *bars = s_bars[w];
    const char *volt = reinterpret_cast<const char *>(tv.volt);
    auto issue_load = [&](int k) {  // lane 0
        const unsigned nr = (unsigned)((wn - k * ST_MT) < ST_MT ? (wn - k * ST_MT) : ST_MT);
        mbar_expect_tx(&bars[k % ST_STAGES], nr * 320u);
        bulk_g2s(ring + (k % ST_STAGES) * ST_STAGE_BYTES, volt + (row0 + (long long)k * ST_MT) * 320, nr * 320u,
                 &bars[k % ST_STAGES]);
    };
    if (lane == 0) {
        for (int st = 0; st < ST_STAGES; ++st) mbar_init(&bars[st], 1);
        for (int k = 0; k < ST_STAGES - 1 && k < nmt; ++k) issue_load(k);
    }
    const int8_t *state = tb.state + row0;
    auto load_states = [&](int r) -> int {      // the state of the warp's row r + lane, -1 if it does not count
        if (r + lane >= wn) return -1;
        const int st = state[r + lane];
        return (row_valid(st, flags) && st >= 0 && st <= 3) ? st : -1;
    };
    // per lane (row rl of a step): nibble j = the state of row 4 j + rl of the 32 (+ 1; 0: the row does
    // not count), bit 3 of the nibble: the 4 rows of step j share one state.  Ten shuffles per 32 rows,
    // away from the steps' critical path (a SHFL + VOTE per step measured ~10 % of the kernel)
    auto pack_states = [&](int v) -> unsigned {
        const int v1 = __shfl_xor_sync(0xffffffffu, v, 1), v2 = __shfl_xor_sync(0xffffffffu, v, 2);
        const bool eq = (v == v1) & (v == v2);           // (no short circuit around a shuffle)
        const unsigned uni = __ballot_sync(0xffffffffu, eq);
        unsigned pk = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int sj = __shfl_sync(0xffffffffu, v, 4 * j + rl);
            pk |= (unsigned)((sj + 1) | ((((uni >> (4 * j)) & 0xfu) == 0xfu) ? 8 : 0)) << (4 * j);
        }
        return pk;
    };
    unsigned st_cur = pack_states(load_states(0));
    int st_next = load_states(32);

    if (threadIdx.x < 128) {   // pivots: |d| at the job's first row of each state
        const int g = threadIdx.x >> 4, dio = (threadIdx.x >> 2) & 3, st = threadIdx.x & 3;
        const int first = jobcnt[JOBCNT * job + 1 + st];
        double pv = 0.0;
        if (first != 0x7fffffff) pv = abs_fast(row_sample(tv, ji.row0 + first, g * 4 + dio));
        s_piv[dio * 4 + st][g] = pv;
    }
    for (int k = threadIdx.x; k < (STATS_THREADS / 32) * NGROUP * STATS_VALS; k += STATS_THREADS)
        (&s_acc[0][0][0])[k] = 0.0;
    double2 off[4];
#pragma unroll
    for (int d = 0; d < 4; ++d) off[d] = tv.offsets ? __ldg(tv.offsets + group * 4 + d) : make_double2(0.0, 0.0);
    __syncthreads();

    int cur = -1;                 // state whose sums the registers hold (warp-uniform)
    double a1[4], a2[4], ac = 0.0;
#pragma unroll
    for (int d = 0; d < 4; ++d) a1[d] = a2[d] = 0.0;
    auto flush = [&]() {
        if (cur < 0) return;
        double v[9] = {ac, a1[0], a1[1], a1[2], a1[3], a2[0], a2[1], a2[2], a2[3]};
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            v[k] += __shfl_xor_sync(0xffffffffu, v[k], 8);
            v[k] += __shfl_xor_sync(0xffffffffu, v[k], 16);
        }
        if (lane < NGROUP) {
            double *acc = s_acc[w][lane];
            acc[cur] += v[0];
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                acc[4 + d * 4 + cur] += v[1 + d];
                acc[20 + d * 4 + cur] += v[5 + d];
            }
        }
        ac = 0.0;
#pragma unroll
        for (int d = 0; d < 4; ++d) a1[d] = a2[d] = 0.0;
    };

    // conflict-free 16-byte reads of a row's 256 diode bytes: groups 0..3 take their first
    // half first, groups 4..7 their second (8 lanes then cover all 32 banks)
    const int hsel = group >> 2;
    int pst = -1;                 // state whose pivots pv[] holds
    double pv[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
    for (int k = 0; k < nmt; ++k) {
        if (k % ST_PER32 == 0 && k > 0) {
            st_cur = pack_states(st_next);
            st_next = load_states((k + ST_PER32) * ST_MT);
        }
        const unsigned char *stage = ring + (k % ST_STAGES) * ST_STAGE_BYTES;
        mbar_wait(&bars[k % ST_STAGES], (unsigned)(k / ST_STAGES) & 1u);
        float4 ra[ST_MT / 4], rb[ST_MT / 4];
#pragma unroll
        for (int hf = 0; hf < ST_MT / 4; ++hf) {
            const unsigned char *q = stage + (hf * 4 + rl) * 320 + 32 * group;
            const float4 u0 = *reinterpret_cast<const float4 *>(q + 16 * hsel);
            const float4 u1 = *reinterpret_cast<const float4 *>(q + 16 * (1 - hsel));
            ra[hf] = hsel ? u1 : u0;
            rb[hf] = hsel ? u0 : u1;
        }
        __syncwarp();            // every lane has read the stage: it can take the load of stage k + 3
        if (lane == 0 && k + ST_STAGES - 1 < nmt) issue_load(k + ST_STAGES - 1);
#pragma unroll
        for (int hf = 0; hf < ST_MT / 4; ++hf) {
            const unsigned nib = (st_cur >> (4 * ((k % ST_PER32) * (ST_MT / 4) + hf))) & 0xfu;
            const int st = (int)(nib & 7u) - 1;
            double x[4] = {0.0, 0.0, 0.0, 0.0};
            if (st >= 0) {
                if (st != pst) {                              // (states come in long runs)
#pragma unroll
                    for (int dio = 0; dio < 4; ++dio) pv[dio] = s_piv[dio * 4 + st][group];
                    pst = st;
                }
                float v[8] = {ra[hf].x, ra[hf].y, ra[hf].z, ra[hf].w, rb[hf].x, rb[hf].y, rb[hf].z, rb[hf].w};
                if (BE) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) v[q] = __uint_as_float(bswap32(__float_as_uint(v[q])));
                }
                double h2[4], ab[4];
#pragma unroll
                for (int dio = 0; dio < 4; ++dio) {
                    const double2 dd = make_double2((double)v[2 * dio] - off[dio].x, (double)v[2 * dio + 1] - off[dio].y);
                    h2[dio] = fma(dd.x, dd.x, dd.y * dd.y);
                }
                sqrt4(h2, ab);
#pragma unroll
                for (int dio = 0; dio < 4; ++dio) x[dio] = ab[dio] - pv[dio];
            }
            if (nib & 8u) {                                   // the usual case: one state (or no valid row)
                const int st0 = st;
                if (st0 >= 0) {
                    if (st0 != cur) { flush(); cur = st0; }
                    ac += 1.0;
#pragma unroll
                    for (int dio = 0; dio < 4; ++dio) {
                        a1[dio] += x[dio];
                        a2[dio] = fma(x[dio], x[dio], a2[dio]);
                    }
                }
            } else {                                          // a run boundary inside the 4 rows
#pragma unroll 1
                for (int s = 0; s < 4; ++s) {
                    if (!__any_sync(0xffffffffu, st == s)) continue;
                    if (s != cur) { flush(); cur = s; }
                    if (st == s) {
                        ac += 1.0;
#pragma unroll
                        for (int dio = 0; dio < 4; ++dio) {
                            a1[dio] += x[dio];
                            a2[dio] = fma(x[dio], x[dio], a2[dio]);
                        }
                    }
                }
            }
        }
    }
    flush();
    __syncthreads();
    for (int k = threadIdx.x; k < NGROUP * STATS_VALS; k += STATS_THREADS) {
        const int g = k / STATS_VALS, v = k - g * STATS_VALS;
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < STATS_THREADS / 32; ++j) sum += s_acc[j][g][v];
        part[((long long)(job * NGROUP + g) * P + p) * STATS_VALS + v] = sum;
    }
}

// add the segments of every (job, group): one thread per (jg, diode, state)
__global__ void k_stats_final(const TableDesc *tabs, const JobInfo *jobs, const int *jobcnt, int njg,
                              int P, const double *part, double *table) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= njg * 16) return;
    const int jg = idx >> 4, ds = idx & 15, st = ds & 3, group = jg & 7;
    const int job = jg >> 3;
    const JobInfo ji = jobs[job];
    const TableDesc &tb = tabs[ji.table];
    if (!tb.state) return;
    const int nseg = stats_segments(ji.nrows);
    double n = 0.0, s1 = 0.0, s2 = 0.0;
    for (int p = 0; p < nseg; ++p) {
        const double *q = part + ((long long)jg * P + p) * STATS_VALS;
        n += q[st];
        s1 += q[4 + ds];
        s2 += q[20 + ds];
    }
    double pv = 0.0;
    const int first = jobcnt[JOBCNT * job + 1 + st];
    if (first != 0x7fffffff) {
        pv = abs_fast(row_sample(tb.tv, ji.row0 + first, group * 4 + (ds >> 2)));
    }
    // mean of an empty state: 0/0 = NaN like Julia's mean of an empty vector;
    // weight = 1 / var = (n - 1) / sum (x - mean)^2   (n == 1 -> 0/0 = NaN as in Julia)
    double2 r;
    r.x = pv + s1 / n;
    r.y = (n - 1.0) / (s2 - s1 * (s1 / n));
    reinterpret_cast<double2 *>(table)[idx] = r;
}

int stats_max_segments(long long max_rows_per_job) { return stats_segments(max_rows_per_job); }

void launch_stats(const Launcher &L, const TableDesc *d_tabs, const JobInfo *d_jobs, int njobs,
                  const int *d_faint_jobs, int nfaint, const int *d_jobcnt, unsigned flags, int P,
                  double *d_part, double *d_table, bool dense) {
    if (nfaint <= 0) return;
    const unsigned grid = (unsigned)((long long)nfaint * P);
    if (dense) {
        cudaFuncSetAttribute(k_stats_seg_bulk<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM);
        cudaFuncSetAttribute(k_stats_seg_bulk<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM);
        if (flags & 16u)
            k_stats_seg_bulk<true><<<grid, STATS_THREADS, ST_SMEM, L.stream>>>(d_tabs, d_jobs, d_faint_jobs, d_jobcnt,
                                                                               flags, P, d_part);
        else
            k_stats_seg_bulk<false><<<grid, STATS_THREADS, ST_SMEM, L.stream>>>(d_tabs, d_jobs, d_faint_jobs, d_jobcnt,
                                                                                flags, P, d_part);
    } else {
        k_stats_seg<<<grid, STATS_THREADS, 0, L.stream>>>(d_tabs, d_jobs, d_faint_jobs, d_jobcnt, flags, P, d_part);
    }
    const int njg = njobs * NGROUP;
    k_stats_final<<<(njg * 16 + 127) / 128, 128, 0, L.stream>>>(d_tabs, d_jobs, d_jobcnt, njg, P, d_part,
                                                               d_table);
    *L.counter += 2;
}

// ===========================================================================
// Demodulation + repack: out = (d [- c]) * exp(-j psi),
//   psi = fl(fl(b sin(fl(theta + phi)) + alpha) - alpha)   over ALL rows
// (reference src/Modulation.jl:417-425, getphase :66-69), then the float32
// re-interleave of src/GPPupilDemodulation.jl:163-171,253.
// ===========================================================================
__device__ __forceinline__ double2 demod_sample(const FitResult &fr, unsigned flags, double theta,
                                                double2 sc, double2 d) {
    PhaseQ pq;
    pq.uniform = fr.uniform; pq.q = fr.q; pq.cq = fr.cq; pq.sq = fr.sq;
    double sn = sin_arg(pq, fr.phi, theta, sc);
    if (!(flags & 4u)) {  // recenter = true
        double gp = __dadd_rn(__dmul_rn(fr.b, sn), fr.alpha);
        double psi = __dadd_rn(gp, -fr.alpha);
        double sp, cp;
        sincos_moderate(psi, &sp, &cp);      // <= 1.5 ulp; falls back to sincos() beyond 1e5
        double vr = d.x, vi = d.y;
        if (flags & 2u) { vr -= fr.cre; vi -= fr.cim; }
        // (vr + j vi) * (cp - j sp)
        return make_double2(__dadd_rn(__dmul_rn(vr, cp), __dmul_rn(vi, sp)),
                            __dadd_rn(__dmul_rn(vi, cp), -__dmul_rn(vr, sp)));
    }
    // recenter = false: data * exp(-1im * angle(model(t))), :424
    double u = __dmul_rn(fr.b, sn);
    double su, cu;
    sincos(u, &su, &cu);
    double mr = __dadd_rn(__dmul_rn(fr.are, cu), -__dmul_rn(fr.aim, su));
    double mi = __dadd_rn(__dmul_rn(fr.are, su), __dmul_rn(fr.aim, cu));
    if (flags & 2u) { mr += fr.cre; mi += fr.cim; }
    double ang = atan2(mi, mr);
    double sa, ca;
    sincos(ang, &sa, &ca);
    return make_double2(__dadd_rn(__dmul_rn(d.x, ca), __dmul_rn(d.y, sa)),
                        __dadd_rn(__dmul_rn(d.y, ca), -__dmul_rn(d.x, sa)));
}

// METROLOGY tables (float32 rows).  Every WARP runs its own pipeline over a contiguous run of
// rows, 8 rows (one mini-tile) at a time, with no block-level synchronisation at all:
//   cp.async.bulk global -> shared into the warp's 3-stage ring (raw rows + basis, tracked by
//   the warp's own mbarriers), results written IN PLACE over the mini-tile, cp.async.bulk
//   shared -> global.  While a warp waits for its bytes the other warps of the SM compute,
//   and the LSU only sees the shared-memory accesses of the arithmetic.  (A copy-only build
//   of this pipeline moves the night at 6.6 TB/s, the measured HBM copy rate.)
// Thread mapping: lane = DIODE (0..31); a warp works on DM_UNROLL rows at a time.  A lane
// reads the 8 bytes of its diode -- a warp reads 256 contiguous bytes, conflict-free -- and
// keeps the constants of its fit (b, alpha, cos q, sin q, c, the centre) in registers for the
// whole job.  The 8 fibre-coupler channels of the 8 rows (128 floats) pass through four per
// lane.  Other layouts (strided / unaligned rows) and keepraw's 144-float rows are staged
// with warp-cooperative word loops through the same buffers.
// complex128 arrays (the demodulateall boundary) are channel-major: there the lanes run
// along the rows (coalesced 16-byte accesses) and a warp loops over the channels.
constexpr int DM_THREADS = 256;
constexpr int DM_WARPS = DM_THREADS / 32;
constexpr int DM_MT = 8;                            // rows per mini-tile
#ifndef DM_WROWS_N
#define DM_WROWS_N 128
#endif
constexpr int DM_WROWS = DM_WROWS_N;                // consecutive rows per warp (16 mini-tiles)
constexpr int DM_BLOCK_ROWS = DM_WARPS * DM_WROWS;  // 1024 rows per block
constexpr int DM_STAGES = 3;
#ifndef DM_UNROLL_N
#define DM_UNROLL_N 1
#endif
constexpr int DM_UNROLL = DM_UNROLL_N;              // rows a warp interleaves
constexpr int DM_STAGE_BYTES = DM_MT * (320 + 16);  // raw rows + basis
constexpr int DM_WARP_BYTES = DM_STAGES * DM_STAGE_BYTES;
constexpr int DM_OUT_BYTES = DM_MT * 144 * 4;       // keepraw staging, per warp
constexpr int DM_SMEM = DM_WARPS * DM_WARP_BYTES;
constexpr int DM_SMEM_KEEPRAW = DM_SMEM + DM_WARPS * DM_OUT_BYTES;
static_assert(DM_MT % DM_UNROLL == 0 && DM_WROWS % DM_MT == 0, "mini-tiles");

// constants of one fit as the demodulation needs them
struct DemodK {
    double b, alpha, cq, sq, cre, cim;
    int uniform;
};
__device__ __forceinline__ DemodK demod_constants(const FitResult *fr, bool offs) {
    const double2 ba = __ldg(reinterpret_cast<const double2 *>(&fr->b));
    const double2 cs = __ldg(reinterpret_cast<const double2 *>(&fr->cq));
    DemodK k;
    k.b = ba.x; k.alpha = ba.y; k.cq = cs.x; k.sq = cs.y;
    k.cre = k.cim = 0.0;
    if (offs) {
        const double2 cc = __ldg(reinterpret_cast<const double2 *>(&fr->cre));
        k.cre = cc.x; k.cim = cc.y;
    }
    k.uniform = __ldg(&fr->uniform);
    return k;
}

// complex128, channel-major (kind 1): lanes along the rows (coalesced 16-byte accesses), a warp
// takes 4 x 32 rows of the block and loops over the channels.  When its rows belong to one job
// with a uniform phase quantum (the usual case) the constants of a fit are loaded once per
// channel and the four rows of a lane are independent chains; psi is a few radians, so the
// sincos_moderate (<= 1.5 ulp) replaces the general-purpose sincos (a third of its instructions).
// The other cases go sample by sample through demod_sample.
__device__ __forceinline__ void demod_arrays_body(const TableDesc &tbg, const FitResult *results, unsigned flags) {
    const TableView &tv = tbg.tv;
    const OutView &ov = tbg.ov;
    const long long n = tv.n, wrows = tbg.wrows;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long blk0 = (long long)blockIdx.x * DM_BLOCK_ROWS;
    const long long blk1 = blk0 + DM_BLOCK_ROWS < n ? blk0 + DM_BLOCK_ROWS : n;
    constexpr int NR = DM_BLOCK_ROWS / DM_THREADS;      // rows per lane
    long long ii[NR];
    bool live[NR];
    double2 sc[NR];
    const long long first = blk0 + warp * 32;
    if (first >= blk1) return;
    long long last = first;
#pragma unroll
    for (int j = 0; j < NR; ++j) {
        const long long i = first + (long long)j * DM_THREADS + lane;
        live[j] = i < blk1;
        ii[j] = live[j] ? i : blk1 - 1;
        sc[j] = tbg.basis[ii[j]];
        const long long wl = first + (long long)j * DM_THREADS + 31;
        if (first + (long long)j * DM_THREADS < blk1) last = wl < blk1 ? wl : blk1 - 1;
    }
    const long long jf = first / wrows;
    const bool onejob = jf == last / wrows;             // warp-uniform
    const bool recenter = !(flags & 4u), offs = (flags & 2u) != 0;
    for (int group = 0; group < NGROUP; ++group) {
        if (!group_on(flags, group)) continue;   // gppd_options.group_mask: columns left untouched
#pragma unroll 1
        for (int dio = 0; dio < 4; ++dio) {
            const int ch = group * 4 + dio;
            const double2 *in = tv.data + (long long)ch * n;
            double2 *out = ov.out + (long long)ch * n;
            bool fast = false;
            DemodK K;
            if (onejob && recenter) {
                K = demod_constants(results + ((long long)tbg.job0 + jf) * NDIODE + ch, offs);
                fast = K.uniform != 0;
            }
            if (fast) {
                double2 d[NR];
#pragma unroll
                for (int j = 0; j < NR; ++j) d[j] = __ldg(in + ii[j]);
#pragma unroll
                for (int j = 0; j < NR; ++j) {
                    // the arithmetic of demod_sample (reference :417-425) with the fit's constants
                    const double sn = fma(sc[j].x, K.cq, sc[j].y * K.sq);
                    const double gp = __dadd_rn(__dmul_rn(K.b, sn), K.alpha);
                    const double psi = __dadd_rn(gp, -K.alpha);
                    double sp, cp;
                    sincos_moderate(psi, &sp, &cp);
                    double vr = d[j].x, vi = d[j].y;
                    if (offs) { vr -= K.cre; vi -= K.cim; }
                    const double2 o = make_double2(__dadd_rn(__dmul_rn(vr, cp), __dmul_rn(vi, sp)),
                                                   __dadd_rn(__dmul_rn(vi, cp), -__dmul_rn(vr, sp)));
                    if (live[j]) out[ii[j]] = o;
                }
            } else {
#pragma unroll
                for (int j = 0; j < NR; ++j) {
                    const FitResult *fr = results + ((long long)tbg.job0 + ii[j] / wrows) * NDIODE + ch;
                    const double2 o = demod_sample(*fr, flags, row_theta(tv, ii[j]), sc[j], row_sample(tv, ii[j], ch));
                    if (live[j]) out[ii[j]] = o;
                }
            }
        }
        const int fcch = fc_channel(group);
#pragma unroll
        for (int j = 0; j < NR; ++j)
            if (live[j]) ov.out[(long long)fcch * n + ii[j]] = __ldg(tv.data + (long long)fcch * n + ii[j]);  // output = copy(data), :353
    }
}

// a batch of complex128 arrays (the f64 entry points) has its own kernel and register budget;
// k_demod keeps an out-of-line copy for a table of that kind inside a mixed batch
__device__ __noinline__ void demod_arrays(const TableDesc &tbg, const FitResult *results, unsigned flags) {
    demod_arrays_body(tbg, results, flags);
}
__global__ void __launch_bounds__(DM_THREADS, 3) k_demod_arrays(const TableDesc *tabs, const FitResult *results,
                                                                unsigned flags) {
    const TableDesc &tbg = tabs[blockIdx.y];
    if ((long long)blockIdx.x * DM_BLOCK_ROWS >= tbg.tv.n) return;
    demod_arrays_body(tbg, results, flags);
}

// BE: raw FITS byte order of the float32 tables (GPPD_BIG_ENDIAN, a batch-wide flag);
// OFFS: the centres are fitted (GPPD_FITOFFSETS): out = (d - c) exp(-j psi)
template <bool BE, bool OFFS>
__global__ void __launch_bounds__(DM_THREADS, 3) k_demod(const TableDesc *tabs, const FitResult *results,
                                                         unsigned flags) {
    const TableDesc &tbg = tabs[blockIdx.y];
    const long long n = tbg.tv.n, wrows = tbg.wrows;
    if ((long long)blockIdx.x * DM_BLOCK_ROWS >= n) return;
    if (tbg.ov.kind == 1) {
        demod_arrays(tbg, results, flags);
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long wr0 = (long long)blockIdx.x * DM_BLOCK_ROWS + (long long)warp * DM_WROWS;
    if (wr0 >= n) return;                      // (no block-level barrier below: a warp may leave)
    const int wn = (int)((n - wr0) < DM_WROWS ? (n - wr0) : DM_WROWS);     // this warp's rows
    const int nmt = (wn + DM_MT - 1) / DM_MT;

    extern __shared__ __align__(128) unsigned char dm_smem[];
    __shared__ uint64_t s_bars[DM_WARPS][DM_STAGES];
    unsigned char *ring = dm_smem + warp * DM_WARP_BYTES;
    uint64_t *bars = s_bars[warp];

    const char *volt_in = reinterpret_cast<const char *>(tbg.tv.volt);
    char *volt_out = reinterpret_cast<char *>(tbg.ov.volt);
    const long long in_stride = tbg.tv.volt_stride, out_stride = tbg.ov.volt_stride;
    const double2 *basis = tbg.basis;
    const double2 *offsets = tbg.tv.offsets;
    const int keepraw = tbg.ov.keepraw;
    const int job0 = tbg.job0, njobs = tbg.njobs;
    const int ow = keepraw ? 144 : 80;   // output words per row
    const int obase = keepraw ? 80 : 0;  // where the demodulated diodes go in an output row
    const bool bulk_in = in_stride == 320 && aligned16(volt_in);
    const bool bulk_out = out_stride == 4 * ow && aligned16(volt_out);
    const bool recenter = !(flags & 4u);
    uint32_t *s_outbuf = reinterpret_cast<uint32_t *>(dm_smem + DM_SMEM + warp * DM_OUT_BYTES);   // keepraw only

    auto mt_rows = [&](int k) { return (wn - k * DM_MT) < DM_MT ? (wn - k * DM_MT) : DM_MT; };
    auto issue_load = [&](int k) {  // lane 0
        const int st = k % DM_STAGES;
        const long long rb = wr0 + (long long)k * DM_MT;
        const unsigned nr = (unsigned)mt_rows(k);
        unsigned char *stage = ring + st * DM_STAGE_BYTES;
        mbar_expect_tx(&bars[st], nr * (320u + 16u));
        bulk_g2s(stage, volt_in + rb * 320, nr * 320u, &bars[st]);
        bulk_g2s(stage + DM_MT * 320, basis + rb, nr * 16u, &bars[st]);
    };
    if (bulk_in) {
        if (lane == 0) {
            for (int st = 0; st < DM_STAGES; ++st) mbar_init(&bars[st], 1);
        }
        __syncwarp();
        if (lane == 0) {
            issue_load(0);
            if (nmt > 1) issue_load(1);
        }
    }

    // this lane's diode: centre of its channel; FC pass-through: floats 4 lane .. 4 lane + 3 of the
    // mini-tile's 8 x 16 FC floats = row lane / 4, FC channels 2 (lane % 4) and 2 (lane % 4) + 1
    const double2 off_d = offsets ? __ldg(offsets + lane) : make_double2(0.0, 0.0);
    const int fc_row = lane >> 2, fc_col = 64 + 4 * (lane & 3);
    const double2 off_f0 = offsets ? __ldg(offsets + NDIODE + 2 * (lane & 3)) : make_double2(0.0, 0.0);
    const double2 off_f1 = offsets ? __ldg(offsets + NDIODE + 2 * (lane & 3) + 1) : make_double2(0.0, 0.0);
    DemodK K;
    K.b = K.alpha = K.cq = K.sq = K.cre = K.cim = 0.0;
    K.uniform = 0;
    long long job_cached = -1;
    if (njobs == 1) {
        K = demod_constants(results + (long long)job0 * NDIODE + lane, OFFS);
        job_cached = 0;
    }

#pragma unroll 1
    for (int k = 0; k < nmt; ++k) {
        const int st = k % DM_STAGES;
        const long long row_base = wr0 + (long long)k * DM_MT;
        const int nrow = mt_rows(k);
        unsigned char *stage = ring + st * DM_STAGE_BYTES;
        uint32_t *s_in = reinterpret_cast<uint32_t *>(stage);
        double2 *s_basis = reinterpret_cast<double2 *>(stage + DM_MT * 320);
        uint32_t *s_out = keepraw ? s_outbuf : s_in;
        if (bulk_in) {
            mbar_wait(&bars[st], (unsigned)(k / DM_STAGES) & 1u);
        } else {
            if (bulk_out) {   // a bulk store of an earlier mini-tile may still be reading this stage
                if (lane == 0) bulk_wait_read();
                __syncwarp();
            }
            for (int w = lane; w < nrow * 80; w += 32) {
                const int r = w / 80, c = w - r * 80;
                s_in[w] = __ldg(reinterpret_cast<const uint32_t *>(volt_in + (row_base + r) * in_stride) + c);
            }
            if (lane < nrow) s_basis[lane] = basis[row_base + lane];
            __syncwarp();
        }
        if (keepraw && k > 0 && bulk_out) {   // the staging buffer is still being read by the last store
            if (lane == 0) bulk_wait_read();
            __syncwarp();
        }

        // one job per mini-tile (the usual case) -> its constants in registers
        bool fast = recenter;
        if (njobs != 1) {
            const long long jf = row_base / wrows, jl = (row_base + nrow - 1) / wrows;
            if (jf != jl) {
                fast = false;
            } else if (jf != job_cached) {
                K = demod_constants(results + ((long long)job0 + jf) * NDIODE + lane, OFFS);
                job_cached = jf;
            }
        }
        // the fast path needs the fit's uniform phase quantum and |psi| <= |b| < 1e4 (sincos_demod);
        // it is taken by the whole warp or not at all, so that it stays straight-line code and
        // the DM_UNROLL rows of an iteration interleave
        fast = fast && K.uniform && fabs(K.b) < 9.0e3;
        const bool wfast = __all_sync(0xffffffffu, fast);

        // FC pass-through first (it reads words that keepraw copies and nobody overwrites)
        uint4 fcw = make_uint4(0u, 0u, 0u, 0u);
        if (!keepraw && fc_row < nrow) {
            fcw = *reinterpret_cast<const uint4 *>(s_in + fc_row * 80 + fc_col);
            uint32_t w[4] = {fcw.x, fcw.y, fcw.z, fcw.w};
            const double o[4] = {off_f0.x, off_f0.y, off_f1.x, off_f1.y};
#pragma unroll
            for (int j = 0; j < 4; ++j) {               // centred FC channel, :170-171
                uint32_t a = w[j];
                if (BE) a = bswap32(a);
                a = __float_as_uint(__double2float_rn((double)__uint_as_float(a) - o[j]));
                if (BE) a = bswap32(a);
                w[j] = a;
            }
            fcw = make_uint4(w[0], w[1], w[2], w[3]);
        }

        if (wfast) {
#pragma unroll 1
            for (int r0 = 0; r0 < nrow; r0 += DM_UNROLL) {
                uint2 raw[DM_UNROLL], res[DM_UNROLL];
                double2 sc[DM_UNROLL];
#pragma unroll
                for (int u = 0; u < DM_UNROLL; ++u) {
                    const int rs = r0 + u < nrow ? r0 + u : r0;     // (rows past the mini-tile repeat row r0)
                    raw[u] = *reinterpret_cast<const uint2 *>(s_in + rs * 80 + 2 * lane);
                    sc[u] = s_basis[rs];
                }
#pragma unroll
                for (int u = 0; u < DM_UNROLL; ++u) {
                    uint32_t a = raw[u].x, b = raw[u].y;
                    if (BE) { a = bswap32(a); b = bswap32(b); }
                    double vr = (double)__uint_as_float(a) - off_d.x;
                    double vi = (double)__uint_as_float(b) - off_d.y;
                    // out = (d - c) exp(-j psi), psi = fl(fl(b sin(theta + q) + alpha) - alpha) = b sin(.)
                    // up to 2 ulp(|psi| + |alpha|) ~ 1e-15, six orders below the float32 result
                    const double sn = fma(sc[u].x, K.cq, sc[u].y * K.sq);
                    const double psi = K.b * sn;
                    double sp, cp;
#ifdef DM_COPY_ONLY     // experiment: the pipeline without the arithmetic
                    sp = 0.0; cp = 1.0 + psi * 1e-300;
#else
                    sincos_demod(psi, &sp, &cp);
#endif
                    if (OFFS) { vr -= K.cre; vi -= K.cim; }
                    a = __float_as_uint(__double2float_rn(fma(vr, cp, vi * sp)));
                    b = __float_as_uint(__double2float_rn(fma(vi, cp, -(vr * sp))));
                    if (BE) { a = bswap32(a); b = bswap32(b); }
                    res[u] = make_uint2(a, b);
                }
#pragma unroll
                for (int u = 0; u < DM_UNROLL; ++u) {
                    const int rr = r0 + u;
                    if (rr >= nrow) continue;
                    if (keepraw) {   // rows 1..80 raw volts, 81..144 demodulated diodes, :163-168
                        const uint32_t *irow = s_in + rr * 80;
                        uint32_t *orow = s_out + rr * 144;
                        orow[lane] = irow[lane];
                        orow[lane + 32] = irow[lane + 32];
                        if (lane < 16) orow[lane + 64] = irow[lane + 64];
                    }
                    *reinterpret_cast<uint2 *>(s_out + rr * ow + obase + 2 * lane) = res[u];
                }
            }
        } else {     // mini-tile straddling two jobs, no uniform quantum, or recenter = false: row by row
#pragma unroll 1
            for (int rr = 0; rr < nrow; ++rr) {
                const uint2 raw = *reinterpret_cast<const uint2 *>(s_in + rr * 80 + 2 * lane);
                uint32_t a = raw.x, b = raw.y;
                if (BE) { a = bswap32(a); b = bswap32(b); }
                const double vr = (double)__uint_as_float(a) - off_d.x;
                const double vi = (double)__uint_as_float(b) - off_d.y;
                const long long i = row_base + rr;
                const FitResult *fr = results + ((long long)job0 + i / wrows) * NDIODE + lane;
                const double2 o = demod_sample(*fr, flags, row_theta(tbg.tv, i), s_basis[rr], make_double2(vr, vi));
                a = __float_as_uint(__double2float_rn(o.x));
                b = __float_as_uint(__double2float_rn(o.y));
                if (BE) { a = bswap32(a); b = bswap32(b); }
                if (keepraw) {
                    const uint32_t *irow = s_in + rr * 80;
                    uint32_t *orow = s_out + rr * 144;
                    orow[lane] = irow[lane];
                    orow[lane + 32] = irow[lane + 32];
                    if (lane < 16) orow[lane + 64] = irow[lane + 64];
                }
                *reinterpret_cast<uint2 *>(s_out + rr * ow + obase + 2 * lane) = make_uint2(a, b);
            }
        }
        if (!keepraw && fc_row < nrow) *reinterpret_cast<uint4 *>(s_out + fc_row * 80 + fc_col) = fcw;

        if (bulk_out) {
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
                bulk_s2g(volt_out + row_base * (4ll * ow), s_out, (unsigned)nrow * 4u * ow);
                bulk_commit();
            }
        } else {
            __syncwarp();
            for (int w = lane; w < nrow * ow; w += 32) {
                const int r = w / ow, c = w - r * ow;
                reinterpret_cast<uint32_t *>(volt_out + (row_base + r) * out_stride)[c] = s_out[w];
            }
            __syncwarp();   // the stage / staging buffer is reused by a later iteration
        }
        // next load: stage (k + 2) % 3 was the stage of mini-tile k - 1, whose store (the group
        // before the one just committed) must have finished reading it
        if (bulk_in && k + 2 < nmt) {
            if (lane == 0) {
                if (bulk_out && !keepraw) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                issue_load(k + 2);
            }
        }
    }
    if (bulk_out && lane == 0) bulk_wait_read();
}

void launch_demod(const Launcher &L, const TableDesc *d_tabs, int ntables, long long max_rows,
                  const FitResult *d_results, unsigned flags, bool arrays) {
    // the 144-float staging buffers are only needed with keepraw (flag bit 8 = GPPD_KEEPRAW)
    const int smem = (flags & 8u) ? DM_SMEM_KEEPRAW : DM_SMEM;
    const dim3 grid((unsigned)((max_rows + DM_BLOCK_ROWS - 1) / DM_BLOCK_ROWS), ntables);
    if (arrays) {          // every table of the batch is a set of complex128 arrays
        k_demod_arrays<<<grid, DM_THREADS, 0, L.stream>>>(d_tabs, d_results, flags);
        *L.counter += 1;
        return;
    }
    const bool be = (flags & 16u) != 0, offs = (flags & 2u) != 0;
#define GPPD_LAUNCH_DEMOD(B, O)                                                                       \
    do {                                                                                              \
        cudaFuncSetAttribute(k_demod<B, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, DM_SMEM_KEEPRAW); \
        k_demod<B, O><<<grid, DM_THREADS, smem, L.stream>>>(d_tabs, d_results, flags);                \
    } while (0)
    if (be && offs) GPPD_LAUNCH_DEMOD(true, true);
    else if (be) GPPD_LAUNCH_DEMOD(true, false);
    else if (offs) GPPD_LAUNCH_DEMOD(false, true);
    else GPPD_LAUNCH_DEMOD(false, false);
#undef GPPD_LAUNCH_DEMOD
    *L.counter += 1;
}

// ===========================================================================
// results -> caller layout: params (c.re,c.im,a.re,a.im,b,phi) with the sign
// normalisation of reference src/Modulation.jl:426-431, chi2, info
// ===========================================================================
__global__ void k_export(const ExportDesc *exps, const FitResult *results, unsigned flags) {
    const ExportDesc &e = exps[blockIdx.y];
    int fl = blockIdx.x * blockDim.x + threadIdx.x;
    if (fl >= e.nfits) return;
    if (!group_on(flags, ((e.fit0 + fl) % NDIODE) >> 2)) return;   // not fitted by this call
    FitResult r = results[e.fit0 + fl];
    double b = r.b, phi = r.phi;
    if (b < 0) {
        b = -b;
        phi += (phi < 0 ? PI_F64 : -PI_F64);
    }
    double *p = e.params + 6ll * fl;
    p[0] = r.cre; p[1] = r.cim; p[2] = r.are; p[3] = r.aim; p[4] = b; p[5] = phi;
    e.chi2[fl] = r.chi2;
    if (e.info) {
        e.info[4 * fl] = r.nfev; e.info[4 * fl + 1] = r.status;
        e.info[4 * fl + 2] = r.method; e.info[4 * fl + 3] = r.second;
    }
}

void launch_export(const Launcher &L, const ExportDesc *d_exps, int ntables, int max_fits,
                   const FitResult *d_results, unsigned flags) {
    k_export<<<dim3((max_fits + 127) / 128, ntables), 128, 0, L.stream>>>(d_exps, d_results, flags);
    *L.counter += 1;
}

// ===========================================================================
// Raw FITS binary-table rows (what FitsUtils.jl's Dict(hdu) / FITScopy! move,
// reference src/FitsUtils.jl:31-37,95-156): records of row_bytes bytes, big-endian,
// TIME (int32) at byte time_off and VOLT (80 float32) at byte volt_off, at any
// alignment.  k_unpack_rows turns them into the dense little-endian TIME / VOLT
// arrays the passes above stream through; k_pack_rows writes the output records:
// the input record with its VOLT field replaced by the 80 (keepraw: 144) output
// floats, every other byte copied.
// ===========================================================================
__device__ __forceinline__ uint32_t load_be32(const unsigned char *p) {
    return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
}

__global__ void k_unpack_rows(const unsigned char *rows, long long n, long long row_bytes,
                              long long time_off, long long volt_off, int32_t *time_us, float *volt) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // (row, word 0..80)
    if (idx >= n * 81) return;
    const long long r = idx / 81;
    const int w = (int)(idx - r * 81);
    const unsigned char *rec = rows + r * row_bytes;
    if (w == 80) time_us[r] = (int32_t)load_be32(rec + time_off);
    else reinterpret_cast<uint32_t *>(volt)[r * 80 + w] = load_be32(rec + volt_off + 4 * w);
}

__global__ void k_pack_rows(const unsigned char *rows, long long n, long long row_bytes,
                            long long volt_off, const float *volt_out, int out_floats,
                            unsigned char *rows_out, long long row_bytes_out) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // output byte
    if (idx >= n * row_bytes_out) return;
    const long long r = idx / row_bytes_out;
    const long long b = idx - r * row_bytes_out;
    const long long vend = volt_off + 4ll * out_floats;
    unsigned char v;
    if (b < volt_off) {
        v = rows[r * row_bytes + b];
    } else if (b < vend) {
        const long long k = b - volt_off;
        const uint32_t word = reinterpret_cast<const uint32_t *>(volt_out)[r * out_floats + (k >> 2)];
        v = (unsigned char)(word >> (8 * (3 - (int)(k & 3))));   // big-endian byte k & 3
    } else {
        v = rows[r * row_bytes + (b - vend) + volt_off + 320];
    }
    rows_out[idx] = v;
}

void launch_unpack_rows(const Launcher &L, const void *d_rows, long long n, long long row_bytes,
                        long long time_off, long long volt_off, int32_t *d_time, float *d_volt) {
    const long long tot = n * 81;
    k_unpack_rows<<<(unsigned)((tot + 255) / 256), 256, 0, L.stream>>>(
        reinterpret_cast<const unsigned char *>(d_rows), n, row_bytes, time_off, volt_off, d_time, d_volt);
    *L.counter += 1;
}

void launch_pack_rows(const Launcher &L, const void *d_rows, long long n, long long row_bytes,
                      long long volt_off, const float *d_volt_out, int out_floats, void *d_rows_out,
                      long long row_bytes_out) {
    const long long tot = n * row_bytes_out;
    k_pack_rows<<<(unsigned)((tot + 255) / 256), 256, 0, L.stream>>>(
        reinterpret_cast<const unsigned char *>(d_rows), n, row_bytes, volt_off, d_volt_out, out_floats,
        reinterpret_cast<unsigned char *>(d_rows_out), row_bytes_out);
    *L.counter += 1;
}

// ===========================================================================
// FP64 unit micro-benchmarks: 16 independent DFMA chains per thread, and 8
// independent mma.sync.m8n8k4.f64 accumulators per warp (the form the harmonic pass
// uses; both run on the same FP64 units).  The larger of the two is the measured
// denominator of the fit's FP64 roofline (MEASURED_PEAKS.json has none).
// ===========================================================================
__global__ void __launch_bounds__(256) k_dfma_peak(double *out, int iters, double a, double b) {
    double x[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) x[k] = (double)(threadIdx.x + k) * 1e-3;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 16; ++k) x[k] = fma(x[k], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += x[k];
    if (s == 12345.678) out[0] = s;  // keep the chains alive
}

__global__ void __launch_bounds__(256) k_dmma_peak(double *out, int iters, double a, double b) {
    double c[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) c[k] = (double)(threadIdx.x + k) * 1e-3;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 8; ++k)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                         : "+d"(c[2 * k]), "+d"(c[2 * k + 1])
                         : "d"(a), "d"(b));
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += c[k];
    if (s == 12345.678) out[0] = s;
}

double measure_dfma_tflops(cudaStream_t stream, double *d_scratch) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int iters = 20000, blocks = sms * 8;
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        const bool mma = rep >= 3;
        cudaEventRecord(a, stream);
        if (mma) k_dmma_peak<<<blocks, 256, 0, stream>>>(d_scratch, iters / 4, 0.999999, 1e-9);
        else k_dfma_peak<<<blocks, 256, 0, stream>>>(d_scratch, iters, 0.999999, 1e-9);
        cudaEventRecord(b, stream);
        cudaEventSynchronize(b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        // one warp-level m8n8k4 = 256 FMAs; one DFMA per thread = 1 FMA
        const double fmas = mma ? 256.0 * 8.0 * (iters / 4) * 8.0 * blocks   // 8 warps per block
                                : 16.0 * iters * 256.0 * blocks;
        const double tf = 2.0 * fmas / (ms * 1e-3) / 1e12;
        if (rep != 0 && rep != 3 && tf > best) best = tf;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return best;
}

}  // namespace gppd
