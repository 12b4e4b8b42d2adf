// Runs the tests of the reference's tester (test/ecostester.cpp of EmbersArc/EiCOS) on the engine:
// fixture headers in the reference's test format (test/**/*.h: data arrays plus a test_<name>()
// that calls ECOS_setup / ECOS_solve / ECOS_updateData / ECOS_cleanup and asserts the exit flag),
// found on the include path under the reference's file names.  tests/test_reference_tester.py
// writes them from the data and expected exit flags stored in tests/golden/fixtures and compiles
// this file against the ECOS-name shim of tests/cpp/shim.  The 18 tests are the ones
// test/ecostester.cpp runs, minus MPC01, whose data the reference does not contain (SURVEY.md F3)
// (infeasible2.h is dead code in the reference: the tester does not include it).  A failed
// mu_assert ends the process, so this main runs ONE named test per process.
// TEST INFRASTRUCTURE: never shipped, never loaded by the product.
#include <cstdio>
#include <cstring>
#include <exception>

#include "minunit.h"
#include "ecos.h"

#include "MPC/MPC02.h"
#include "updateData/update_data.h"
#include "cvxpyProblems/githubIssue98.h"
#include "feasibilityProblems/feas.h"
#include "unboundedProblems/unboundedLP1.h"
#include "infeasibleProblems/infeasible1.h"
#include "unboundedProblems/unboundedMaxSqrt.h"
#include "emptyProblem/emptyProblem.h"
#include "LPnetlib/lp_25fv47.h"
#include "LPnetlib/lp_adlittle.h"
#include "LPnetlib/lp_afiro.h"
#include "LPnetlib/lp_agg.h"
#include "LPnetlib/lp_agg2.h"
#include "LPnetlib/lp_agg3.h"
#include "LPnetlib/lp_bandm.h"
#include "LPnetlib/lp_beaconfd.h"
#include "LPnetlib/lp_blend.h"
#include "LPnetlib/lp_bnl1.h"

namespace
{
struct Entry
{
    const char *name;
    char *(*fn)();
};
const Entry TESTS[] = {
    {"MPC02", test_MPC02}, {"update_data", test_update_data}, {"unboundedLP1", test_unboundedLP1},
    {"unboundedMaxSqrt", test_unboundedMaxSqrt}, {"feas", test_feas}, {"infeasible1", test_infeasible1},
    {"lp_25fv47", test_lp_25fv47}, {"lp_adlittle", test_lp_adlittle},
    {"lp_afiro", test_lp_afiro}, {"lp_agg", test_lp_agg}, {"lp_agg2", test_lp_agg2}, {"lp_agg3", test_lp_agg3},
    {"lp_bandm", test_lp_bandm}, {"lp_beaconfd", test_lp_beaconfd}, {"lp_blend", test_lp_blend},
    {"lp_bnl1", test_lp_bnl1}, {"emptyProblem", test_emptyProblem}, {"issue98", test_issue98},
};
} // namespace

int main(int argc, char **argv)
{
    if (argc < 2)
    {
        for (const Entry &e : TESTS)
            printf("%s\n", e.name);
        return 0;
    }
    for (const Entry &e : TESTS)
        if (!strcmp(e.name, argv[1]))
        {
            try
            {
                char *msg = e.fn(); // mu_assert ends the process when the expectation fails
                if (msg)
                {
                    printf("FAIL %s: %s\n", e.name, msg);
                    return 1;
                }
            }
            catch (const std::exception &ex)
            {
                printf("ERROR %s: %s\n", e.name, ex.what());
                return 2;
            }
            printf("PASS %s\n", e.name);
            return 0;
        }
    printf("unknown test %s\n", argv[1]);
    return 3;
}
