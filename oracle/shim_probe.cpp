// shim_probe.cpp -- C entry points into the stand-in third-party headers of ref_shim/ (mini_cv.h, mini_eigen.h) themselves, so that
// tests can pin THEM against cv2 fixtures and numpy (tests/test_ref_pin.py).  TEST INFRASTRUCTURE (oracle/).  Built on its own into
// _build/libshim.so: it needs none of the reference's sources.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "Eigen/Dense"
#include "opencv2/opencv.hpp"

extern "C" {
// cv::remap as Tracking::pred_patch_fc calls it (src/Tracking.cpp:272): CV_32F source and maps, INTER_LINEAR, BORDER_CONSTANT 0
void ref_cv_remap(const float* src, int srows, int scols, const float* mapx, const float* mapy, int orows, int ocols, float* dst) {
    cv::Mat s(srows, scols, CV_32F, (void*)src, (size_t)scols * 4), mx(orows, ocols, CV_32F, (void*)mapx, (size_t)ocols * 4),
        my(orows, ocols, CV_32F, (void*)mapy, (size_t)ocols * 4), out;
    cv::remap(s, out, mx, my, cv::INTER_LINEAR, 0, cvScalarAll(0));
    for (int i = 0; i < orows; i++)
        for (int j = 0; j < ocols; j++) dst[i * ocols + j] = out.at<float>(i, j);
}
// cv::calcCovarMatrix as Converter::corrcoef_opencv calls it (src/Converter.cpp:195): CV_32F samples, one per row (np x nv, row-major),
// CV_COVAR_NORMAL | CV_COVAR_ROWS, CV_64F scatter matrix about the mean (nv x nv, row-major)
void ref_cv_calc_covar(const float* M_rowmajor, int np, int nv, double* out_rowmajor) {
    cv::Mat M(np, nv, CV_32F, (void*)M_rowmajor, (size_t)nv * 4), cov, mean;
    cv::calcCovarMatrix(M, cov, mean, CV_COVAR_NORMAL | CV_COVAR_ROWS, CV_64F);
    for (int i = 0; i < nv; i++)
        for (int j = 0; j < nv; j++) out_rowmajor[(size_t)i * nv + j] = cov.at<double>(i, j);
}
// cv::FAST(img, kps, threshold, nonmax), keypoints in output order
int ref_cv_fast(const uint8_t* img, int rows, int cols, int threshold, int nonmax, int max_kp, int* xy) {
    cv::Mat im(rows, cols, CV_8U, (void*)img, (size_t)cols);
    std::vector<cv::KeyPoint> kp;
    cv::FAST(im, kp, threshold, nonmax != 0);
    for (size_t i = 0; i < kp.size() && (int)i < max_kp; i++) {
        xy[2 * i] = (int)kp[i].pt.x;
        xy[2 * i + 1] = (int)kp[i].pt.y;
    }
    return (int)kp.size();
}
// Eigen semantics the reference's sources depend on, evaluated by the stand-in; tests compare with numpy (tests/test_ref_pin.py).
// in: A (n x n, column-major), v (n).  out: see the test for the layout.
int ref_eigen_probe(const double* A_colmajor, const double* v_in, int n, double* out, int out_cap) {
    using namespace Eigen;
    std::vector<double> o;
    auto push = [&](const MatrixXd& m) {  // column-major dump
        for (Index j = 0; j < m.cols(); j++)
            for (Index i = 0; i < m.rows(); i++) o.push_back(m(i, j));
    };
    std::vector<double> a_buf(A_colmajor, A_colmajor + (size_t)n * n);  // Eigen::Map<MatrixXd> wants a non-const pointer
    MatrixXd A = Eigen::Map<MatrixXd>(a_buf.data(), n, n);
    VectorXd v(n);
    for (int i = 0; i < n; i++) v(i) = v_in[i];
    // 1. comma initialiser fills row by row, whatever the storage order (the Q16 pattern, src/Map.cpp:379)
    Matrix<double, 3, 2> c32;
    c32 << 1, 2, 3, 4, 5, 6;
    push(c32);
    // 2. block-row comma initialisation (src/Map.cpp:397 pattern): [A11 A12; A21 A22] from four blocks, then vector stacking
    MatrixXd blk(n, n);
    blk << A.topLeftCorner(2, 2), A.topRightCorner(2, n - 2), A.bottomLeftCorner(n - 2, 2), A.bottomRightCorner(n - 2, n - 2);
    push(blk);
    VectorXd st(n + 2);
    st << v.head(2), 7.0, v.tail(n - 2), 9.0;
    push(st);
    // 3. dynamic inverse (partial-pivot LU) and fixed-size inverse (cofactors)
    push(A.inverse());
    Matrix3d A3 = A.topLeftCorner(3, 3);
    push(A3.inverse());
    Matrix2d A2 = A.block(1, 1, 2, 2);
    push(A2.inverse());
    // 4. views alias their parent; vector <-> row-vector assignment transposes
    MatrixXd B = A;
    B.block(1, 1, 2, 2) = MatrixXd::Identity(2, 2) * 5.0;
    B.col(0).head(2) << -1, -2;
    B.middleRows(2, 1).col(3) = MatrixXd::Ones(1, 1) * 42.0;
    push(B);
    RowVectorXd rv = v;
    VectorXd back = rv;
    push(rv);
    push(back);
    // 5. array expressions as ExtendKF::distort_fm writes them (src/ExtendKF.cpp:185-203)
    MatrixXd r1 = A.row(0), r2 = A.row(1);
    MatrixXd ru = (r1.array().pow(2) + r2.array().pow(2)).array().sqrt();
    MatrixXd rd = ru.array() / (1 + 0.06333 * ru.array().pow(2) + 0.0139 * ru.array().pow(4));
    push(rd);
    // 6. 1 x 1 products convert to scalars; left-to-right products; asDiagonal
    const double quad = v.transpose() * A * v;
    o.push_back(quad);
    push(A * v.asDiagonal());
    // 7. maxCoeff(&idx): first maximum; a NaN in slot 0 is sticky
    VectorXd mc(5);
    mc << 1, 7, 3, 7, 2;
    double idx = -1;
    o.push_back(mc.maxCoeff(&idx));
    o.push_back(idx);
    mc(0) = std::nan("");
    o.push_back(mc.maxCoeff(&idx));
    o.push_back(idx);
    // 8. self-adjoint eigenvalues (ascending), as Tracking::matching uses them on S (src/Tracking.cpp:301)
    MatrixXd S2 = A.topLeftCorner(2, 2) * A.topLeftCorner(2, 2).transpose();
    SelfAdjointEigenSolver<MatrixXd> es(S2);
    push(es.eigenvalues());
    // 9. Map as a column-major reshape; resize keeps the data when the element count is unchanged
    MatrixXd rs = Eigen::Map<MatrixXd>(A.data(), n * n / 2, 2);
    push(rs);
    MatrixXd keep = A;
    keep.resize(n * n, 1);
    push(keep);
    // 10. (array < t).rowwise().count() (src/Tracking.cpp:476)
    Matrix<ptrdiff_t, Dynamic, Dynamic> cnt = (A.array() < 0.5).rowwise().count();
    for (Index i = 0; i < cnt.rows(); i++) o.push_back((double)cnt(i));
    // 11. cross / norm / segment on a row vector
    Vector3d a3 = v.head(3), b3 = v.segment(2, 3);
    push(a3.cross(b3));
    o.push_back(v.norm());
    push(rv.segment(1, 3));
    if ((int)o.size() > out_cap) return -(int)o.size();
    std::memcpy(out, o.data(), sizeof(double) * o.size());
    return (int)o.size();
}
}  // extern "C"
