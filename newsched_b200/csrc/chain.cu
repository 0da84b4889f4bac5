// chain.cu -- back-to-back execution of op handles on device buffers, and the host-buffer
// streaming driver (H2D / compute / D2H overlapped on three streams).
//
// This is what a host-resident source -> [device blocks] -> host-resident sink costs end to
// end: the analogue of the reference's H2D -> D2D -> D2H edge chain
// (schedulers/mt/test/cuda/qa_scheduler_mt_cuda_copy.cpp:36-38, runtime/lib/cudabuffer.cu:126-158)
// without its per-call stream synchronisation and mirror copies.
#include <vector>

#include "common.cuh"

using namespace b200;

namespace {

struct stage {
    b200_chain_op op;
    int in_item_bytes = 0;  // bytes per input item of this stage (sample granularity)
    int out_item_bytes = 0;
    long long num = 1, den = 1; // out_items = in_items * num / den
    long long multiple = 1;     // in_items must be a multiple of this
};

constexpr int NSLOT = 3;

} // namespace

struct b200_chain {
    std::vector<stage> stages;
    int in_item_bytes = 0;
    long long chunk_items = 0;
    std::vector<long long> stage_in_items; // per stage, for a full chunk
    void* d_tmp[2] = { nullptr, nullptr };
    size_t tmp_bytes = 0;
    // host streaming resources (lazy)
    bool host_ready = false;
    cudaStream_t st_in = nullptr, st_c = nullptr, st_out = nullptr;
    void* d_in[NSLOT] = { nullptr, nullptr, nullptr };
    void* d_out[NSLOT] = { nullptr, nullptr, nullptr };
    cudaEvent_t ev_in[NSLOT], ev_c[NSLOT], ev_free[NSLOT], ev_in_free[NSLOT];
    size_t chunk_in_bytes = 0, chunk_out_bytes = 0;
};

static int stage_describe(stage& st, int in_bytes)
{
    st.in_item_bytes = in_bytes;
    switch (st.op.kind) {
    case B200_OP_COPY:
        st.out_item_bytes = in_bytes;
        break;
    case B200_OP_MULTIPLY_CONST_CC:
        if (in_bytes != 8)
            return set_err(B200_ERR_ARG, "chain: multiply_const_cc needs complex64 items");
        st.out_item_bytes = 8;
        break;
    case B200_OP_MULTIPLY_CONST_FF:
        if (in_bytes != 4)
            return set_err(B200_ERR_ARG, "chain: multiply_const_ff needs float items");
        st.out_item_bytes = 4;
        break;
    case B200_OP_COMPLEX_TO_MAG:
        if (in_bytes != 8)
            return set_err(B200_ERR_ARG, "chain: complex_to_mag needs complex64 items");
        st.out_item_bytes = 4;
        break;
    default:
        return set_err(B200_ERR_ARG, "chain: unknown op kind %d", st.op.kind);
    }
    return B200_OK;
}

static int run_stage(const stage& st, const void* in, void* out, long long n_items,
                     long long* n_out_items, cudaStream_t s)
{
    b200_stream_t bs = reinterpret_cast<b200_stream_t>(s);
    int rc = B200_OK;
    switch (st.op.kind) {
    case B200_OP_COPY:
        rc = b200_copy(out, in, (size_t)n_items * st.in_item_bytes, bs);
        *n_out_items = n_items;
        break;
    case B200_OP_MULTIPLY_CONST_CC:
        rc = b200_multiply_const_cc(out, in, st.op.k_re, st.op.k_im, (size_t)n_items, bs);
        *n_out_items = n_items;
        break;
    case B200_OP_MULTIPLY_CONST_FF:
        rc = b200_multiply_const_ff((float*)out, (const float*)in, st.op.k_re, (size_t)n_items, bs);
        *n_out_items = n_items;
        break;
    case B200_OP_COMPLEX_TO_MAG:
        rc = b200_complex_to_mag((float*)out, in, (size_t)n_items, bs);
        *n_out_items = n_items;
        break;
    case B200_OP_FIR: {
        int64_t nc = 0, np = 0;
        rc = b200_fir_run((b200_fir*)st.op.handle, in, out, n_items, &nc, &np, bs);
        if (rc == B200_OK && nc != n_items)
            return set_err(B200_ERR_ARG, "chain: fir stage left %lld items unconsumed",
                           (long long)(n_items - nc));
        *n_out_items = np;
        break;
    }
    case B200_OP_FFT: {
        if (n_items % st.multiple)
            return set_err(B200_ERR_ARG, "chain: fft stage needs a multiple of N items");
        rc = b200_fft_run((b200_fft*)st.op.handle, in, out, n_items / st.multiple, bs);
        *n_out_items = n_items;
        break;
    }
    case B200_OP_PFB: {
        int64_t nc = 0, nv = 0;
        rc = b200_pfb_run((b200_pfb*)st.op.handle, in, out, n_items, &nc, &nv, bs);
        if (rc == B200_OK && nc != n_items)
            return set_err(B200_ERR_ARG, "chain: pfb stage left items unconsumed");
        *n_out_items = n_items * st.num / st.den;
        break;
    }
    default:
        return set_err(B200_ERR_ARG, "chain: unknown op kind %d", st.op.kind);
    }
    return rc;
}

extern "C" {

int b200_chain_destroy(b200_chain* c)
{
    if (!c)
        return B200_OK;
    cudaFree(c->d_tmp[0]);
    cudaFree(c->d_tmp[1]);
    if (c->host_ready) {
        for (int i = 0; i < NSLOT; i++) {
            cudaFree(c->d_in[i]);
            cudaFree(c->d_out[i]);
            cudaEventDestroy(c->ev_in[i]);
            cudaEventDestroy(c->ev_c[i]);
            cudaEventDestroy(c->ev_free[i]);
            cudaEventDestroy(c->ev_in_free[i]);
        }
        cudaStreamDestroy(c->st_in);
        cudaStreamDestroy(c->st_c);
        cudaStreamDestroy(c->st_out);
    }
    delete c;
    return B200_OK;
}

int b200_chain_create(const b200_chain_op* ops, int32_t n_ops, int32_t in_item_bytes,
                      int64_t chunk_items, b200_chain** out)
{
    if (!ops || n_ops < 1 || !out || in_item_bytes < 1 || chunk_items < 1)
        return set_err(B200_ERR_ARG, "chain_create: bad argument");
    *out = nullptr;
    b200_chain* c = new b200_chain();
    c->in_item_bytes = in_item_bytes;
    c->chunk_items = chunk_items;
    int bytes = in_item_bytes;
    long long items = chunk_items;
    size_t max_mid = 0;
    for (int i = 0; i < n_ops; i++) {
        stage st;
        st.op = ops[i];
        int rc = B200_OK;
        if (st.op.kind == B200_OP_FIR) {
            int d = 1, ib = 0;
            rc = b200_fir_geometry((b200_fir*)st.op.handle, &d, &ib);
            if (rc == B200_OK && ib != bytes)
                rc = set_err(B200_ERR_ARG, "chain: fir item size %d != upstream %d", ib, bytes);
            st.in_item_bytes = bytes;
            st.out_item_bytes = bytes;
            st.num = 1;
            st.den = d;
            st.multiple = d;
        } else if (st.op.kind == B200_OP_FFT) {
            int n = 0, ob = 0;
            rc = b200_fft_geometry((b200_fft*)st.op.handle, &n, &ob);
            if (rc == B200_OK && bytes != 8)
                rc = set_err(B200_ERR_ARG, "chain: fft needs complex64 items");
            st.in_item_bytes = 8;
            st.out_item_bytes = ob;
            st.multiple = n;
        } else if (st.op.kind == B200_OP_PFB) {
            int m = 0, cc = 0;
            int32_t os = 1;
            rc = b200_pfb_geometry((b200_pfb*)st.op.handle, &m, &cc);
            if (rc == B200_OK)
                rc = b200_pfb_get_oversample((b200_pfb*)st.op.handle, &os);
            if (rc == B200_OK && bytes != 8)
                rc = set_err(B200_ERR_ARG, "chain: pfb needs complex64 items");
            st.in_item_bytes = 8;
            st.out_item_bytes = 8;
            st.num = cc; // cc channels out per hop of D = M / oversample items in
            st.den = m / os;
            st.multiple = m / os;
        } else {
            rc = stage_describe(st, bytes);
        }
        if (rc == B200_OK && items % st.multiple)
            rc = set_err(B200_ERR_ARG, "chain_create: chunk_items does not divide evenly at stage %d", i);
        if (rc != B200_OK) {
            delete c;
            return rc;
        }
        c->stage_in_items.push_back(items);
        items = items * st.num / st.den;
        bytes = st.out_item_bytes;
        if (i + 1 < n_ops) {
            size_t b = (size_t)items * bytes;
            if (b > max_mid)
                max_mid = b;
        }
        c->stages.push_back(st);
    }
    c->chunk_in_bytes = (size_t)chunk_items * in_item_bytes;
    c->chunk_out_bytes = (size_t)items * bytes;
    c->tmp_bytes = max_mid;
    if (max_mid) {
        for (int i = 0; i < 2; i++) {
            cudaError_t e = cudaMalloc(&c->d_tmp[i], max_mid);
            if (e != cudaSuccess) {
                b200_chain_destroy(c);
                return set_err(B200_ERR_NOMEM, "chain_create: cudaMalloc(%zu) -> %s", max_mid,
                               cudaGetErrorString(e));
            }
        }
    }
    *out = c;
    return B200_OK;
}

int64_t b200_chain_out_bytes_bound(const b200_chain* c, int64_t n_in_items)
{
    if (!c)
        return -1;
    long long items = n_in_items;
    int bytes = c->in_item_bytes;
    for (const stage& st : c->stages) {
        items = items * st.num / st.den;
        bytes = st.out_item_bytes;
    }
    return items * bytes;
}

// one chunk (n_items <= chunk_items) through all stages on stream s
static int chain_chunk(b200_chain* c, const void* d_in, void* d_out, long long n_items,
                       long long* out_bytes, cudaStream_t s)
{
    const void* cur = d_in;
    long long items = n_items;
    int bytes = c->in_item_bytes;
    const int n = (int)c->stages.size();
    for (int i = 0; i < n; i++) {
        const stage& st = c->stages[i];
        if (items % st.multiple)
            return set_err(B200_ERR_ARG, "chain_run: %lld items do not divide evenly at stage %d",
                           items, i);
        void* dst = (i == n - 1) ? d_out : c->d_tmp[i & 1];
        long long no = 0;
        int rc = run_stage(st, cur, dst, items, &no, s);
        if (rc != B200_OK)
            return rc;
        items = no;
        bytes = st.out_item_bytes;
        cur = dst;
    }
    *out_bytes = items * bytes;
    return B200_OK;
}

int b200_chain_run(b200_chain* c, const void* d_in, void* d_out, int64_t n_in_items,
                   int64_t* n_out_bytes, b200_stream_t s)
{
    if (!c || n_in_items < 0 || (n_in_items > 0 && (!d_in || !d_out)))
        return set_err(B200_ERR_ARG, "chain_run: bad argument");
    long long done = 0, outb = 0;
    while (done < n_in_items) {
        long long n = n_in_items - done < c->chunk_items ? n_in_items - done : c->chunk_items;
        long long ob = 0;
        int rc = chain_chunk(c, (const char*)d_in + done * c->in_item_bytes, (char*)d_out + outb, n,
                             &ob, cs(s));
        if (rc != B200_OK)
            return rc;
        done += n;
        outb += ob;
    }
    if (n_out_bytes)
        *n_out_bytes = outb;
    return B200_OK;
}

static int chain_host_init(b200_chain* c)
{
    if (c->host_ready)
        return B200_OK;
    B200_CUDA(cudaStreamCreateWithFlags(&c->st_in, cudaStreamNonBlocking));
    B200_CUDA(cudaStreamCreateWithFlags(&c->st_c, cudaStreamNonBlocking));
    B200_CUDA(cudaStreamCreateWithFlags(&c->st_out, cudaStreamNonBlocking));
    for (int i = 0; i < NSLOT; i++) {
        B200_CUDA(cudaMalloc(&c->d_in[i], c->chunk_in_bytes));
        B200_CUDA(cudaMalloc(&c->d_out[i], c->chunk_out_bytes ? c->chunk_out_bytes : 1));
        B200_CUDA(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
        B200_CUDA(cudaEventCreateWithFlags(&c->ev_c[i], cudaEventDisableTiming));
        B200_CUDA(cudaEventCreateWithFlags(&c->ev_free[i], cudaEventDisableTiming));
        B200_CUDA(cudaEventCreateWithFlags(&c->ev_in_free[i], cudaEventDisableTiming));
    }
    c->host_ready = true;
    return B200_OK;
}

int b200_chain_run_host(b200_chain* c, const void* h_in, void* h_out, int64_t n_in_items,
                        int64_t* n_out_bytes)
{
    if (!c || n_in_items < 0 || (n_in_items > 0 && (!h_in || !h_out)))
        return set_err(B200_ERR_ARG, "chain_run_host: bad argument");
    int rc = chain_host_init(c);
    if (rc != B200_OK)
        return rc;
    long long done = 0, outb = 0;
    long long k = 0;
    while (done < n_in_items) {
        long long n = n_in_items - done < c->chunk_items ? n_in_items - done : c->chunk_items;
        int slot = (int)(k % NSLOT);
        if (k >= NSLOT) {
            // the slot's device input is free once its compute finished, its device output
            // once its D2H finished
            B200_CUDA(cudaStreamWaitEvent(c->st_in, c->ev_in_free[slot], 0));
            B200_CUDA(cudaStreamWaitEvent(c->st_c, c->ev_free[slot], 0));
        }
        B200_CUDA(cudaMemcpyAsync(c->d_in[slot], (const char*)h_in + done * c->in_item_bytes,
                                  (size_t)n * c->in_item_bytes, cudaMemcpyHostToDevice, c->st_in));
        B200_CUDA(cudaEventRecord(c->ev_in[slot], c->st_in));
        B200_CUDA(cudaStreamWaitEvent(c->st_c, c->ev_in[slot], 0));
        long long ob = 0;
        rc = chain_chunk(c, c->d_in[slot], c->d_out[slot], n, &ob, c->st_c);
        if (rc != B200_OK) {
            cudaDeviceSynchronize();
            return rc;
        }
        B200_CUDA(cudaEventRecord(c->ev_c[slot], c->st_c));
        B200_CUDA(cudaEventRecord(c->ev_in_free[slot], c->st_c));
        B200_CUDA(cudaStreamWaitEvent(c->st_out, c->ev_c[slot], 0));
        B200_CUDA(cudaMemcpyAsync((char*)h_out + outb, c->d_out[slot], (size_t)ob,
                                  cudaMemcpyDeviceToHost, c->st_out));
        B200_CUDA(cudaEventRecord(c->ev_free[slot], c->st_out));
        done += n;
        outb += ob;
        k++;
    }
    B200_CUDA(cudaStreamSynchronize(c->st_out));
    B200_CUDA(cudaStreamSynchronize(c->st_c));
    if (n_out_bytes)
        *n_out_bytes = outb;
    return B200_OK;
}

} // extern "C"
