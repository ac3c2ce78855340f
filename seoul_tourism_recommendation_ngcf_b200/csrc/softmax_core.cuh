// The launches of the in-batch softmax loss (softmax_loss.cu), shared with the cosine InfoNCE (xsimgcl.cu).
#pragma once
#include "common.cuh"

struct SoftmaxRun {
    const float *u, *p, *n;        // rows, columns p (then n; NULL: none)
    int64_t batch;
    int D;
    const int64_t *pos_ids, *neg_ids;
    float temperature, weight_decay, batch_size;
    // optional validity flags [batch] (0 / 1): a row outside them has no loss term and a zero gradient row, and a column
    // outside them is masked for every row; the loss is then divided by the number of valid rows (not batch_size), whose
    // inverse goes to *inv_count, and G is left unscaled by it (g_scale = 1 / temperature with batch_size = 1)
    const uint8_t* valid;
    float* inv_count;
    float *loss, *gu, *gp, *gn;    // gu NULL: forward only
};

// bytes of the (1024-byte-aligned) workspace softmax_run needs
size_t softmax_run_bytes(int64_t batch, bool has_n, int D);
// the launches on `ws`, 1024-byte aligned; arguments already checked by the caller
int softmax_run(const SoftmaxRun& r, uint8_t* ws, cudaStream_t st);
