// A getInput() input plug-in for the driver's `--inpLibA L A` (the plug-in ABI of the reference driver, src/geneo4PETSc.cpp:75-96):
// an irregular graph Laplacian of --size N nodes (N >= 8).  A ring of edges, chords i -- (7 i + 3) mod N and a triangle
// every fifth node, each element weighted 1 + (e mod 5) / 4, --inpEps E (default 1e-4) on the diagonal of every element.
// Compiled by tests/test_host.py into a temporary directory.
#include <set>
#include <sstream>
#include <string>
#include <vector>

extern "C" int getInput(std::string const& args, unsigned int& nbElem, unsigned int& nbNode, std::vector<unsigned int>& elemPtr,
                        std::vector<unsigned int>& elemIdx, std::vector<std::vector<double>>& elemSubMat) {
  unsigned int n = 0;
  double eps = 1e-4;
  std::istringstream in(args);
  for (std::string tok; in >> tok;) {
    if (tok == "--size") in >> n;
    else if (tok == "--inpEps") in >> eps;
    else return 1;
  }
  if (n < 8) return 1;
  std::vector<std::vector<unsigned int>> elems;
  std::set<std::pair<unsigned int, unsigned int>> edges;
  auto edge = [&](unsigned int a, unsigned int b) {
    if (a != b && edges.insert({a < b ? a : b, a < b ? b : a}).second) elems.push_back({a, b});
  };
  for (unsigned int i = 0; i < n; i++) edge(i, (i + 1) % n);
  for (unsigned int i = 0; i < n; i++) edge(i, (unsigned int)((7ull * i + 3) % n));
  for (unsigned int i = 0; i + 4 < n; i += 5) elems.push_back({i, i + 2, i + 4});
  nbNode = n;
  nbElem = (unsigned int)elems.size();
  elemPtr.assign(1, 0);
  elemIdx.clear();
  elemSubMat.clear();
  for (size_t e = 0; e < elems.size(); e++) {
    const std::vector<unsigned int>& d = elems[e];
    const size_t k = d.size();
    const double w = 1.0 + (double)(e % 5) / 4.0;
    std::vector<double> m(k * k);
    for (size_t r = 0; r < k; r++)
      for (size_t c = 0; c < k; c++) m[r * k + c] = r == c ? w * (double)(k - 1) + eps : -w;
    elemIdx.insert(elemIdx.end(), d.begin(), d.end());
    elemPtr.push_back((unsigned int)elemIdx.size());
    elemSubMat.push_back(m);
  }
  return 0;
}
