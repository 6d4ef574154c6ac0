// matvec.cu -- host side of the decode matvec: launch plan, workspace sizing, per-format dispatch.
// The kernel lives in matvec_impl.cuh and is instantiated per format in inst_<format>.cu.
#include <cstdlib>

#include "matvec_common.cuh"

namespace b200q {

static cudaError_t launch_family(int family, const MatvecParams& p, int mb, int grid, int smem, cudaStream_t st) {
    switch (family) {
        case B200Q_FAM_Q4_K: return mv_launch<B200Q_FAM_Q4_K>(p, mb, grid, smem, st);
        case B200Q_FAM_Q6_K: return mv_launch<B200Q_FAM_Q6_K>(p, mb, grid, smem, st);
        case B200Q_FAM_Q8_0: return mv_launch<B200Q_FAM_Q8_0>(p, mb, grid, smem, st);
        case B200Q_FAM_Q5_K: return mv_launch<B200Q_FAM_Q5_K>(p, mb, grid, smem, st);
        case B200Q_FAM_Q4_1: return mv_launch<B200Q_FAM_Q4_1>(p, mb, grid, smem, st);
        case B200Q_FAM_Q5_1: return mv_launch<B200Q_FAM_Q5_1>(p, mb, grid, smem, st);
        case B200Q_FAM_Q2_K: return mv_launch<B200Q_FAM_Q2_K>(p, mb, grid, smem, st);
        case B200Q_FAM_Q3_K: return mv_launch<B200Q_FAM_Q3_K>(p, mb, grid, smem, st);
        case B200Q_FAM_IQ4_XS: return mv_launch<B200Q_FAM_IQ4_XS>(p, mb, grid, smem, st);
        case B200Q_FAM_TQ2_0: return mv_launch<B200Q_FAM_TQ2_0>(p, mb, grid, smem, st);
        case B200Q_FAM_I8S: return mv_launch<B200Q_FAM_I8S>(p, mb, grid, smem, st);
        case B200Q_FAM_G4: return mv_launch<B200Q_FAM_G4>(p, mb, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}
static long long* g_trace = nullptr;
static int g_trace_launch = 0;
void set_matvec_trace(long long* p) { g_trace = p; g_trace_launch = 0; }

// dual-format partner honoured by a launch: plain / norm-prologue matvecs only (not the SwiGLU, grouped or fused-exchange forms)
static const b200q_weight* dual_partner(const b200q_weight* w) { return w->pair; }

cudaError_t matvec_plan(const b200q_weight* w, int64_t M, MatvecPlan* plan, int pro) {
    if (M < 1 || M > 4) return cudaErrorInvalidValue;
    int mb = M == 1 ? 1 : (M == 2 ? 2 : 4);
    const b200q_weight* w2 = dual_partner(w);
    const int cbmax = (w2 && w2->chunk_bytes > w->chunk_bytes) ? w2->chunk_bytes : w->chunk_bytes;
    int stage = cbmax + (pro ? 0 : (int)M * ACT_REC_BYTES);
    stage = (stage + 127) & ~127;
    int xhat = pro ? (int)(((size_t)w->KC * M * ACT_REC_BYTES + 127) & ~(size_t)127) : 0;
    // > half an SM on purpose: two CTAs of one launch must never share an SM (measured: after glue kernels perturb
    // the placement, doubled-up CTAs run at half speed and the launch takes 2x); cross-launch overlap is done
    // with the L2 prefetch kernel instead
    int budget_kb = 150;
    if (const char* e = getenv("B200Q_MV_SMEM_KB")) { int v = atoi(e); if (v >= 64 && v <= 214) budget_kb = v; }
    int budget = budget_kb * 1024 - MV_HDR_BYTES - xhat;
    int nst = budget / stage;
    if (nst > MV_MAX_STAGES) nst = MV_MAX_STAGES;
    if (const char* e = getenv("B200Q_MV_STAGES")) { int v = atoi(e); if (v >= 2 && v < nst) nst = v; }
    if (nst < 2) return cudaErrorInvalidValue;
    int64_t C = (w->T + (w2 ? w2->T : 0)) * w->KC;
    int64_t G = (int64_t)w->num_sms;
    if (const char* e = getenv("B200Q_MV_GRID")) { int v = atoi(e); if (v >= 1 && v <= w->num_sms) G = v; }  // ws_part holds num_sms slots
    if (G > C) G = C;
    plan->grid = (int)G;
    plan->nstages = nst;
    plan->stage_bytes = stage;
    plan->smem_bytes = MV_HDR_BYTES + xhat + nst * stage;
    plan->xhat_bytes = xhat;
    plan->mb = mb;
    return cudaSuccess;
}

size_t matvec_ws_bytes(const b200q_weight* w, int64_t M) {
    // counters (one per row tile, padded) + 2 partial slots per potential CTA
    size_t cnt = ((size_t)w->T * 4 + 255) & ~(size_t)255;
    size_t part = (size_t)w->num_sms * 2 * TILE_ROWS * 4 * sizeof(double);
    (void)M;
    return cnt + part;
}

cudaError_t launch_matvec(const b200q_weight* w, const uint8_t* xq, int64_t M, void* y, int y_dtype, int64_t ldy, uint8_t* ws, cudaStream_t st,
                          const FusedPrologue* fp, const RemoteOut* ro, void* swiglu_xq_out) {
    MatvecPlan plan;
    const int pro = fp ? fp->mode : 0;
    const b200q_weight* w2 = dual_partner(w);
    // a paired weight is launched together with its partner, by the plain / norm-prologue forms only; y holds N1 + N2 columns
    if (w2 && (ro || swiglu_xq_out || (fp && fp->mode != 1) || ldy < w->N + w2->N)) return cudaErrorInvalidValue;
    cudaError_t e = matvec_plan(w, M, &plan, pro);
    if (e != cudaSuccess) return e;
    MatvecParams p;
    p.w = w->data;
    p.xq = xq;
    p.y = y;
    p.bias = w->bias;
    size_t cnt = ((size_t)w->T * 4 + 255) & ~(size_t)255;
    p.ws_cnt = reinterpret_cast<unsigned int*>(ws);
    p.ws_part = reinterpret_cast<double*>(ws + cnt);
    p.N = w->N + (w2 ? w2->N : 0);       // dual: rows of w2 follow (N1 % 128 == 0, checked by b200q_weight_set_pair)
    p.M = (int)M;
    p.y_dtype = y_dtype;
    p.ldy = ldy;
    p.KC = w->KC;
    p.C = (w->T + (w2 ? w2->T : 0)) * w->KC;
    p.gpc = w->gpc;
    p.nstages = plan.nstages;
    p.chunk_bytes = (w2 && w2->chunk_bytes > w->chunk_bytes) ? w2->chunk_bytes : w->chunk_bytes;
    p.cb1 = w->chunk_bytes;
    p.cb2 = w2 ? w2->chunk_bytes : 0;
    p.w2 = w2 ? w2->data : nullptr;
    p.T1 = (int)w->T;
    p.gpc2 = w2 ? w2->gpc : 0;
    p.stage_bytes = plan.stage_bytes;
    p.pro = pro;
    p.xhat_bytes = plan.xhat_bytes;
    p.h_in = fp ? fp->h_in : nullptr;
    p.delta = fp ? fp->delta : nullptr;
    p.h_out = fp ? fp->h_out : nullptr;
    p.norm_w = fp ? fp->norm_w : nullptr;
    p.eps = fp ? fp->eps : 0.0f;
    p.gate_up = fp ? fp->gate_up : nullptr;
    p.w_table = nullptr;
    p.sel = nullptr;
    p.n_experts = 0;
    p.tpw = (int)(w->T + (w2 ? w2->T : 0));
    p.x_rows = (int)M;
    p.x_slot_div = 1;
    p.y_slot_stride = 0;
    p.trace = g_trace ? g_trace + (size_t)(g_trace_launch++) * 148 * 8 : nullptr;
    p.debug_flags = 0;
    p.xq_out = (uint8_t*)swiglu_xq_out;
    p.epi_F = (int)(w->N / 2);
    p.epi_rows = (int)M;
    p.plan32 = ((p.C + 1) * (int64_t)plan.grid < (1ll << 32)) ? 1 : 0;
    p.rp_mode = ro ? ro->mode : RP_NONE;
    if (ro) p.comm = ro->comm;
    else p.comm = CommDev{};
    p.next_w = nullptr;
    p.next_C = p.next_KC = 0;
    p.next_chunk_bytes = p.next_G = p.next_pf = 0;
    if (w->next && w->next->device == w->device && !pro) {
        // successor prefetch budget: what HBM can deliver during this launch's tail + the boundary (~6 us ~ 40 MB), well
        // inside the 126 MB L2.  B200Q_MV_NEXT_PF_MB overrides (0 disables).
        static const double pf_mb = [] { const char* e = getenv("B200Q_MV_NEXT_PF_MB"); return e ? atof(e) : 32.0; }();
        MatvecPlan np_;
        if (pf_mb > 0 && matvec_plan(w->next, M, &np_, 0) == cudaSuccess) {
            const int64_t per_cta = (int64_t)(pf_mb * 1048576.0) / ((int64_t)np_.grid * w->next->chunk_bytes);
            if (per_cta >= 1) {
                p.next_w = w->next->data;
                p.next_C = w->next->T * w->next->KC;
                p.next_KC = w->next->KC;
                p.next_chunk_bytes = w->next->chunk_bytes;
                p.next_G = np_.grid;
                p.next_pf = per_cta > 4096 ? 4096 : (int)per_cta;
            }
        }
    }
    {
        // L2 prefetch budget: at most ~64 MB per launch so a huge weight (lm_head) cannot thrash the 126 MB L2
        int64_t per_cta = (64ll << 20) / ((int64_t)plan.grid * p.chunk_bytes);
        p.l2_prefetch_chunks = 0;  // measured: prefetching into L2 from here delays the x copy and slows the predecessor (r1 notes)
        (void)per_cta;
        if (const char* e = getenv("B200Q_MV_L2PF")) p.l2_prefetch_chunks = atoi(e);
    }
    if (const char* e = getenv("B200Q_MV_DEBUG")) p.debug_flags = atoi(e);
    if (w2) {
        p.next_w = nullptr; p.next_pf = 0;
        if (w->family == B200Q_FAM_Q4_K && w2->family == B200Q_FAM_Q6_K) return mv_launch_dual_q4k_q6k(p, plan.mb, plan.grid, plan.smem_bytes, st);
        return cudaErrorInvalidValue;
    }
    return launch_family(w->family, p, plan.mb, plan.grid, plan.smem_bytes, st);
}

// ---- grouped launch over an expert bank: n_slots independent M = 1 matvecs in one stream-K grid ----
size_t matvec_grouped_ws_bytes(const b200q_bank* b, int64_t n_slots) {
    size_t cnt = ((size_t)b->proto.T * (size_t)n_slots * 4 + 255) & ~(size_t)255;
    size_t part = (size_t)b->proto.num_sms * 2 * TILE_ROWS * 4 * sizeof(double);
    return cnt + part;
}

cudaError_t launch_matvec_grouped(const b200q_bank* b, const int32_t* sel_dev, int64_t n_slots, const uint8_t* xq, int64_t x_rows, int64_t x_slot_div,
                                  void* y, int y_dtype, int64_t y_slot_stride, uint8_t* ws, cudaStream_t st, void* swiglu_xq_out) {
    b200q_weight v = b->proto;  // virtual weight: the selected experts' tiles back to back
    v.T = b->proto.T * n_slots;
    MatvecPlan plan;
    cudaError_t e = matvec_plan(&v, 1, &plan, 0);
    if (e != cudaSuccess) return e;
    if (plan.stage_bytes - (v.chunk_bytes + ACT_REC_BYTES) < 16) return cudaErrorInvalidValue;  // room for the per-stage skip flag
    MatvecParams p = {};
    p.w = nullptr;
    p.xq = xq;
    p.y = y;
    p.bias = nullptr;
    size_t cnt = ((size_t)v.T * 4 + 255) & ~(size_t)255;
    p.ws_cnt = reinterpret_cast<unsigned int*>(ws);
    p.ws_part = reinterpret_cast<double*>(ws + cnt);
    p.N = b->proto.N;
    p.M = 1;
    p.y_dtype = y_dtype;
    p.ldy = b->proto.N;
    p.KC = v.KC;
    p.C = v.T * v.KC;
    p.gpc = v.gpc;
    p.nstages = plan.nstages;
    p.chunk_bytes = v.chunk_bytes;
    p.stage_bytes = plan.stage_bytes;
    p.w_table = b->table_dev;
    p.sel = sel_dev;
    p.n_experts = b->E;
    p.w2 = nullptr; p.cb1 = v.chunk_bytes; p.cb2 = 0; p.T1 = 0; p.gpc2 = 0;
    p.tpw = (int)b->proto.T;
    p.x_rows = (int)x_rows;
    p.x_slot_div = (int)x_slot_div;
    p.y_slot_stride = y_slot_stride;
    p.next_w = nullptr;
    p.next_pf = 0;
    p.xq_out = (uint8_t*)swiglu_xq_out;
    p.epi_F = (int)(b->proto.N / 2);
    p.epi_rows = (int)n_slots;
    p.plan32 = ((p.C + 1) * (int64_t)plan.grid < (1ll << 32)) ? 1 : 0;
    return launch_family(v.family, p, 1, plan.grid, plan.smem_bytes, st);
}

}  // namespace b200q
