// double_hoisting_driver.cpp -- b200::Linear_Transform_Plain_double_hoisted from C++ through seal/seal.h: the diagonals are
// encoded at context->key_parms_id(), the result must decrypt to U v within 1e-4.  Prints "DOUBLE HOISTED OK" on success.
#include <cmath>
#include <cstdlib>
#include <iostream>

#include "ckks_b200_helper.h"

using namespace seal;
using namespace std;

int main() {
    EncryptionParameters params(scheme_type::CKKS);
    const size_t n = 8192;
    params.set_poly_modulus_degree(n);
    params.set_coeff_modulus(CoeffModulus::Create(n, {60, 40, 40, 60}));
    auto context = SEALContext::Create(params);
    KeyGenerator keygen(context);
    Encryptor encryptor(context, keygen.public_key());
    Decryptor decryptor(context, keygen.secret_key());
    CKKSEncoder encoder(context);
    const double scale = pow(2.0, 40);
    const int d = 16;
    vector<int> steps{-d};
    for (int l = 1; l < d; l++) steps.push_back(l);
    GaloisKeys gk = keygen.galois_keys(steps);
    srand(11);
    auto rnd = [] { return (double)rand() / RAND_MAX; };
    vector<vector<double>> U(d, vector<double>(d));
    vector<double> v(d);
    for (auto &row : U)
        for (auto &x : row) x = rnd();
    for (auto &x : v) x = rnd();
    vector<Plaintext> diag_pt(d);
    for (int l = 0; l < d; l++) {   // diag_l[k] = U[k][(k + l) mod d]
        vector<double> diag(d);
        for (int k = 0; k < d; k++) diag[k] = U[k][(k + l) % d];
        encoder.encode(diag, context->key_parms_id(), scale, diag_pt[l]);
    }
    Plaintext pv;
    encoder.encode(v, scale, pv);
    Ciphertext cv;
    encryptor.encrypt(pv, cv);
    Ciphertext got = b200::Linear_Transform_Plain_double_hoisted(cv, diag_pt, gk, params);
    Plaintext p;
    vector<double> out;
    decryptor.decrypt(got, p);
    encoder.decode(p, out);
    double err = 0;
    for (int i = 0; i < d; i++) {
        double want = 0;
        for (int j = 0; j < d; j++) want += U[i][j] * v[j];
        err = max(err, fabs(out[i] - want));
    }
    cout << "b200::Linear_Transform_Plain_double_hoisted (d = " << d << "): max |decrypt - U v| = " << err << endl;
    bool rejected = false;   // diagonals at the ciphertext level are refused
    try {
        vector<Plaintext> low(1);
        encoder.encode(v, scale, low[0]);
        b200::Linear_Transform_Plain_double_hoisted(cv, low, gk, params);
    } catch (const invalid_argument &) {
        rejected = true;
    }
    if (err < 1e-4 && rejected) cout << "DOUBLE HOISTED OK" << endl;
    return err < 1e-4 && rejected ? 0 : 1;
}
