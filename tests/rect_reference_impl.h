/* TEST INFRASTRUCTURE ONLY -- included by rect_reference.c once per element type (T, FN as in oracle/svd_oracle.c). */
/* qr_apply_q of the oracle (A += Q2^T A, svd_cpu.h:345-353) with the loops in the order k, i, c: every P[i][c] is still
 * 0 + the products for k = 0, 1, ... added one at a time, so the result is the same to the bit, but the inner loop runs
 * along rows of A and P (the oracle's order walks columns of Q2 and A and makes tall panels take minutes). */
static void FN(rect_apply_q)(T* A, size_t lda, size_t rows, size_t cols, const T* Q2, T* P) {
    memset(P, 0, sizeof(T) * rows * cols);
    for (size_t k = 0; k < rows; ++k)
        for (size_t i = 0; i < rows; ++i) {
            const T q = Q2[k * rows + i];
            for (size_t c = 0; c < cols; ++c) P[i * cols + c] += q * A[k * lda + c];
        }
    for (size_t i = 0; i < rows; ++i)
        for (size_t c = 0; c < cols; ++c) A[i * lda + c] = A[i * lda + c] + P[i * cols + c];
}

int FN(rect_brd_p1_panel_mn)(T* A, size_t mrows, size_t n, size_t b) {
    if (b == 0 || n == 0 || n % b != 0 || mrows < n) return -1;
    T* S = (T*)calloc(b * b, sizeof(T));
    for (size_t k = 0; k < n; k += b) {
        size_t m = mrows - k;                  /* trailing rows */
        size_t nc = n - k - b;                 /* trailing cols right of the panel */
        T* V = (T*)calloc(m * b, sizeof(T));
        T* work = (T*)calloc(b * b + 2 * m * b + m + 2 * b + 16, sizeof(T));
        FN(qr)(A + k * n + k, n, m, b, S, b, V, b, work);
        free(work);
        if (nc > 0) {
            T* Q1 = (T*)malloc(sizeof(T) * (b * m + m * m));
            T* Q2 = Q1 + b * m;
            FN(form_q)(Q2, S, b, V, b, m, b, Q1);
            T* P = (T*)malloc(sizeof(T) * m * nc);
            FN(rect_apply_q)(A + k * n + k + b, n, m, nc, Q2, P);
            free(P); free(Q1);
        }
        free(V);
        if (k + b < n - 1) {
            size_t mr = m - b;                 /* rows below the row panel */
            T* U = (T*)calloc(b * nc, sizeof(T));
            T* work2 = (T*)calloc(b * b + 3 * b * nc + nc + 2 * b + 16, sizeof(T));
            FN(lq)(A + k * n + k + b, n, b, nc, S, b, U, nc, work2);
            free(work2);
            if (mr > 0) {
                T* P1 = (T*)malloc(sizeof(T) * (b * nc + nc * nc));
                T* Pm = P1 + b * nc;
                FN(form_p)(Pm, S, b, U, nc, nc, b, P1);
                T* R = (T*)malloc(sizeof(T) * mr * nc);
                FN(lq_apply_p)(A + (k + b) * n + k + b, n, mr, nc, Pm, R);
                free(R); free(P1);
            }
            free(U);
        }
    }
    free(S);
    return 0;
}
