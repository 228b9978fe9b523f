// matmul_blocked_driver.cpp -- b200::CC_Matrix_Multiplication_blocked from C++ through seal/seal.h at d = 4 on a 2 x 3 by
// 3 x 2 tile grid: every output tile must be bit-identical to the sum over l of b200::CC_Matrix_Multiplication(A_il, B_lj)
// added with Evaluator::add, and decrypt to the tile of A B.  Prints "MATMUL BLOCKED OK" on success.
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <iostream>

#include "ckks_b200_helper.h"

using namespace seal;
using namespace std;

static vector<uint64_t> words(const Ciphertext &ct) {   // the active limbs of every polynomial, on the host
    const auto &p = ct.poly();
    const size_t n = p.eng->n;
    vector<uint64_t> out((size_t)p.size * p.limbs * n);
    for (int k = 0; k < p.size; k++)
        seal::detail::check(ckks_download(p.eng->ctx, out.data() + (size_t)k * p.limbs * n, p.buf->p + (size_t)k * p.cap * n,
                                          (size_t)p.limbs * n * 8, nullptr));
    return out;
}

int main() {
    EncryptionParameters params(scheme_type::CKKS);
    const size_t n = 8192;
    params.set_poly_modulus_degree(n);
    params.set_coeff_modulus(CoeffModulus::Create(n, {60, 40, 40, 40, 40, 60}));   // the config-4 chain
    auto context = SEALContext::Create(params);
    KeyGenerator keygen(context);
    Encryptor encryptor(context, keygen.public_key());
    Decryptor decryptor(context, keygen.secret_key());
    CKKSEncoder encoder(context);
    const double scale = pow(2.0, 40), eps = 1e-8;
    const int d = 4, dd = d * d, tn = 2, tm = 3, tp = 2;
    vector<int> steps;
    for (int i = 0; i < 12; i++) steps.push_back(1 << i), steps.push_back(-(1 << i));   // |step| < N/2
    GaloisKeys gk = keygen.galois_keys(steps);
    // the permutation matrices of eprint 2018/1041 as diagonals (diag_l[k] = U[k][(k + l) mod d^2]), + epsilon
    auto diagonals = [&](auto col) {   // col(i, j): the column of row d i + j's one
        vector<vector<double>> U(dd, vector<double>(dd, 0.0));
        for (int i = 0; i < d; i++)
            for (int j = 0; j < d; j++) U[d * i + j][col(i, j)] = 1.0;
        vector<Plaintext> pts(dd);
        for (int l = 0; l < dd; l++) {
            vector<double> diag(dd);
            for (int k = 0; k < dd; k++) diag[k] = U[k][(k + l) % dd] + eps;
            encoder.encode(diag, scale, pts[l]);
        }
        return pts;
    };
    vector<Plaintext> sigma = diagonals([&](int i, int j) { return d * i + (i + j) % d; });
    vector<Plaintext> tau = diagonals([&](int i, int j) { return d * ((i + j) % d) + j; });
    vector<vector<Plaintext>> V, W;
    for (int k = 1; k < d; k++) {
        V.push_back(diagonals([&](int i, int j) { return d * i + (j + k) % d; }));
        W.push_back(diagonals([&](int i, int j) { return d * ((i + k) % d) + j; }));
    }
    srand(21);
    auto rnd = [] { return (double)rand() / RAND_MAX; };
    vector<vector<double>> A(tn * d, vector<double>(tm * d)), B(tm * d, vector<double>(tp * d));
    for (auto &r : A)
        for (auto &x : r) x = rnd();
    for (auto &r : B)
        for (auto &x : r) x = rnd();
    auto tile = [&](const vector<vector<double>> &M, int r, int c) {
        vector<double> v(dd);
        for (int i = 0; i < d; i++)
            for (int j = 0; j < d; j++) v[d * i + j] = M[r * d + i][c * d + j];
        Plaintext p;
        encoder.encode(v, scale, p);
        Ciphertext ct;
        encryptor.encrypt(p, ct);
        return ct;
    };
    vector<Ciphertext> At, Bt;
    for (int i = 0; i < tn; i++)
        for (int l = 0; l < tm; l++) At.push_back(tile(A, i, l));
    for (int l = 0; l < tm; l++)
        for (int j = 0; j < tp; j++) Bt.push_back(tile(B, l, j));
    vector<Ciphertext> got = b200::CC_Matrix_Multiplication_blocked(At, Bt, tn, tm, tp, d, sigma, tau, V, W, gk, params);
    Evaluator evaluator(context);
    bool same = got.size() == (size_t)(tn * tp);
    double err = 0;
    for (int i = 0; i < tn && same; i++) {
        for (int j = 0; j < tp; j++) {
            Ciphertext want = b200::CC_Matrix_Multiplication(At[i * tm], Bt[j], d, sigma, tau, V, W, gk, params);
            for (int l = 1; l < tm; l++) {
                Ciphertext p = b200::CC_Matrix_Multiplication(At[i * tm + l], Bt[l * tp + j], d, sigma, tau, V, W, gk, params);
                evaluator.add_inplace(want, p);
            }
            const Ciphertext &g = got[i * tp + j];
            same = same && g.poly().size == 3 && g.poly().limbs == want.poly().limbs && g.scale() == want.scale() &&
                   words(g) == words(want);
            Plaintext pt;
            vector<double> out;
            decryptor.decrypt(g, pt);
            encoder.decode(pt, out);
            for (int r = 0; r < d; r++)
                for (int c = 0; c < d; c++) {
                    double ab = 0;
                    for (int k = 0; k < tm * d; k++) ab += A[i * d + r][k] * B[k][j * d + c];
                    err = max(err, fabs(out[d * r + c] - ab));
                }
        }
    }
    cout << "b200::CC_Matrix_Multiplication_blocked (d = " << d << ", " << tn << " x " << tm << " x " << tp
         << " tiles): bit-identical to the per-tile sum: " << same << ", max |decrypt - A B| = " << err << endl;
    bool rejected = false;
    try {
        b200::CC_Matrix_Multiplication_blocked(At, Bt, tn, tm + 1, tp, d, sigma, tau, V, W, gk, params);
    } catch (const invalid_argument &) {
        rejected = true;
    }
    const bool ok = same && err < 1e-3 && rejected;
    if (ok) cout << "MATMUL BLOCKED OK" << endl;
    return ok ? 0 : 1;
}
