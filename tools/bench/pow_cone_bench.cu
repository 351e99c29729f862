// Times cone_pow_kernel (the kernel conic_setup launches for power cones) on K cones of random v and random exponents,
// and reports the evaluations of psi per cone.  Usage: pow_cone_bench K [reps] -> one JSON line.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <random>
#include <vector>

#include "../../diffopt.jl_b200/csrc/pow_cone.cuh"

#define CK(x)                                                                       \
    do {                                                                            \
        cudaError_t e_ = (x);                                                       \
        if (e_ != cudaSuccess) {                                                    \
            fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); \
            return 1;                                                               \
        }                                                                           \
    } while (0)

int main(int argc, char** argv) {
    const int K = argc > 1 ? atoi(argv[1]) : 100000;
    const int reps = argc > 2 ? atoi(argv[2]) : 20;
    std::mt19937_64 gen(7);
    std::normal_distribution<double> nd;
    std::uniform_real_distribution<double> ud(-3.0, 2.0), ua(0.05, 0.95);
    std::vector<double> v(3 * (size_t)K), alpha(K);
    std::vector<int> off(K);
    std::vector<signed char> neg(K);
    for (int c = 0; c < K; ++c) {
        const double sc = pow(10.0, ud(gen));
        for (int k = 0; k < 3; ++k) v[3 * (size_t)c + k] = nd(gen) * sc;
        alpha[c] = ua(gen);
        off[c] = 3 * c;
        neg[c] = (signed char)(c & 1);
    }
    double *dv, *dvp, *dblk, *dal;
    int *doff, *dit;
    signed char* dneg;
    CK(cudaMalloc(&dv, sizeof(double) * v.size()));
    CK(cudaMalloc(&dvp, sizeof(double) * v.size()));
    CK(cudaMalloc(&dblk, sizeof(double) * 3 * v.size()));
    CK(cudaMalloc(&dal, sizeof(double) * K));
    CK(cudaMalloc(&doff, sizeof(int) * K));
    CK(cudaMalloc(&dit, sizeof(int) * K));
    CK(cudaMalloc(&dneg, K));
    CK(cudaMemcpy(dv, v.data(), sizeof(double) * v.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dal, alpha.data(), sizeof(double) * K, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(doff, off.data(), sizeof(int) * K, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dneg, neg.data(), K, cudaMemcpyHostToDevice));
    int sms = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    int blocks = (K + 127) / 128;   // as conic_setup launches it
    if (blocks > sms * 16) blocks = sms * 16;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    cone_pow_kernel<<<blocks, 128>>>(K, doff, dneg, dal, dv, dvp, dblk, dit);   // warm-up, and the counts
    CK(cudaDeviceSynchronize());
    std::vector<int> it(K);
    CK(cudaMemcpy(it.data(), dit, sizeof(int) * K, cudaMemcpyDeviceToHost));
    CK(cudaEventRecord(e0));
    for (int r = 0; r < reps; ++r) cone_pow_kernel<<<blocks, 128>>>(K, doff, dneg, dal, dv, dvp, dblk, nullptr);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    long long sum = 0, n4 = 0;
    int mx = 0;
    for (int c = 0; c < K; ++c) {
        if (it[c] > 0) { sum += it[c]; ++n4; }
        mx = it[c] > mx ? it[c] : mx;
    }
    printf("{\"cones\": %d, \"kernel_ms\": %.5f, \"case4_fraction\": %.4f, \"psi_evals_max\": %d, \"psi_evals_mean_case4\": %.3f}\n",
           K, ms / reps, (double)n4 / K, mx, n4 ? (double)sum / n4 : 0.0);
    cudaFree(dv); cudaFree(dvp); cudaFree(dblk); cudaFree(dal); cudaFree(doff); cudaFree(dit); cudaFree(dneg);
    return 0;
}
