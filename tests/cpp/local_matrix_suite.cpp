// C++ port of the reference's LocalMatrixSuite (src/test/scala/edu/nju/pasalab/marlin/matrix/LocalMatrixSuite.scala),
// written against the compiled host mirror include/marlin_b200.hpp.  The expected values are the suite's own literals
// (small integers: every assertion is exact).  Needs a B200; without one the first call throws the library's
// "no CPU fallback" error and the program exits with status 3.
#include "marlin_b200.hpp"

#include <cstdio>
#include <functional>

using namespace marlin;
using BDM = DenseMatrix;

static int failures = 0, passed = 0;
#define CHECK(cond)                                                                                       \
    do {                                                                                                  \
        if (!(cond)) { std::printf("  FAILED %s:%d  %s\n", __FILE__, __LINE__, #cond); ++failures; }     \
    } while (0)

static void test(const char* name, const std::function<void()>& body) {
    const int before = failures;
    try { body(); } catch (const std::exception& e) { std::printf("  EXCEPTION in '%s': %s\n", name, e.what()); ++failures; }
    if (failures == before) ++passed;
    std::printf("[%s] %s\n", failures == before ? " ok " : "FAIL", name);
}

// :10-13 — the sparse matrix every case uses, one SparseVector per column
static SparseMatrix spMat() {
    return SparseMatrix(4, 4, {{4, {1}, {1.0}}, {4, {0, 3}, {2.0, 1.0}}, {4, {0}, {3.0}}, {4, {2}, {4.0}}});
}
static BDM deMat() { return BDM{{0.0, 1.0, 2.0, 3.0}, {2.0, 3.0, 4.0, 5.0}, {3.0, 2.0, 1.0, 0.0}, {1.0, 1.0, 1.0, 1.0}}; }

int main() {
    try {
        Context::get();
    } catch (const std::exception& e) {
        std::printf("%s\n", e.what());
        return 3;
    }
    test("sparse matrix to breeze `DenseMatrix`", [] {                                       // :8-21
        const BDM expected{{0.0, 2.0, 3.0, 0.0}, {1.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 4.0}, {0.0, 1.0, 0.0, 0.0}};
        CHECK(spMat().toDense().denseBlock() == expected);
    });
    test("breeze `DenseMatrix` multiply sparse matrix", [] {                                 // :23-40
        const BDM expected{{1.0, 3.0, 0.0, 8.0}, {3.0, 9.0, 6.0, 16.0}, {2.0, 6.0, 9.0, 4.0}, {1.0, 3.0, 3.0, 4.0}};
        CHECK(LibMatrixMult::multDenseSparse(SubMatrix(deMat()), spMat()).denseBlock() == expected);
    });
    test("sparse matrix multiply sparse matrix", [] {                                        // :42-53
        const BDM expected{{2.0, 0.0, 0.0, 12.0}, {0.0, 2.0, 3.0, 0.0}, {0.0, 4.0, 0.0, 0.0}, {1.0, 0.0, 0.0, 0.0}};
        CHECK(spMat().multiply(spMat()).denseBlock() == expected);
    });
    test("sparse matrix multiply breeze `DenseMatrix`", [] {                                 // :55-72
        const BDM expected{{13.0, 12.0, 11.0, 10.0}, {0.0, 1.0, 2.0, 3.0}, {4.0, 4.0, 4.0, 4.0}, {2.0, 3.0, 4.0, 5.0}};
        CHECK(LibMatrixMult::multSparseDense(spMat(), SubMatrix(deMat())).denseBlock() == expected);
    });
    test("sparse SubMatrix dispatch and refusals (SubMatrix.scala:41-139)", [] {
        SubMatrix s(spMat()), d(deMat());
        CHECK(s.isSparse() && !d.isSparse() && s.rows() == 4 && s.cols() == 4);
        CHECK(s.multiply(d).denseBlock() == LibMatrixMult::multSparseDense(spMat(), d).denseBlock());
        // scalar ops map the stored values only: implicit zeros stay zero
        const BDM plus1{{0.0, 3.0, 4.0, 0.0}, {2.0, 0.0, 0.0, 0.0}, {0.0, 0.0, 0.0, 5.0}, {0.0, 2.0, 0.0, 0.0}};
        CHECK(s.add(1.0).denseBlock() == plus1);
        CHECK(s.multiply(2.0).divide(2.0).denseBlock() == spMat().toDense().denseBlock());
        bool threw = false;
        try { s.add(d); } catch (const std::invalid_argument&) { threw = true; }
        CHECK(threw);
        threw = false;
        try { SparseMatrix(4, 2, {{4, {2, 1}, {1.0, 1.0}}, {4, {}, {}}}); } catch (const std::invalid_argument&) { threw = true; }
        CHECK(threw);                                                                         // unsorted rows refused
    });
    std::printf("%d passed, %d failed checks\n", passed, failures);
    return failures == 0 ? 0 : 1;
}
