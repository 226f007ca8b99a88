// driver.cpp -- drives the REFERENCE's own compiler half (IR + CKKS passes +
// reference executor, compiled from /root/reference where it lies; see
// build.sh and SURVEY.md Appendix C) to produce golden fixtures:
//   stdin : a program in the little text format written by tests/golden/gen_golden.py
//   stdout: JSON with the compiled term list, parameters and signature.
// Test infrastructure only (oracle/_ref); never shipped or linked by the product.
#include "eva/ckks/ckks_compiler.h"
#include "eva/common/program_traversal.h"
#include "eva/common/reference_executor.h"
#include "eva/ir/program.h"
#include <cstdio>
#include <iostream>
#include <map>
#include <sstream>
#include <string>
using namespace eva;

static std::string jstr(const std::string &s) { return "\"" + s + "\""; }

struct Dumper {
  Program &p;
  TermMap<Type> types;
  std::ostringstream out;
  bool first = true;
  Dumper(Program &p) : p(p), types(p) {}
  void operator()(const Term::Ptr &t) {
    out << (first ? "" : ",\n") << "  {\"id\":" << t->index << ",\"op\":" << jstr(getOpName(t->op)) << ",\"args\":[";
    first = false;
    bool f = true;
    for (auto &o : t->getOperands()) { out << (f ? "" : ",") << o->index; f = false; }
    out << "]";
    if (t->has<TypeAttribute>()) out << ",\"type\":" << jstr(getTypeName(t->get<TypeAttribute>()));
    if (t->has<RotationAttribute>()) out << ",\"rotation\":" << t->get<RotationAttribute>();
    if (t->has<RescaleDivisorAttribute>()) out << ",\"divisor\":" << t->get<RescaleDivisorAttribute>();
    if (t->has<EncodeAtScaleAttribute>()) out << ",\"scale\":" << t->get<EncodeAtScaleAttribute>();
    if (t->has<EncodeAtLevelAttribute>()) out << ",\"level\":" << t->get<EncodeAtLevelAttribute>();
    if (t->has<RangeAttribute>()) out << ",\"range\":" << t->get<RangeAttribute>();
    if (t->has<ConstantValueAttribute>()) {
      std::vector<double> v;
      t->get<ConstantValueAttribute>()->expandTo(v, p.getVecSize());
      bool uniform = true;
      for (auto x : v) if (x != v[0]) uniform = false;
      out << ",\"const\":[";
      char buf[64];
      size_t n = uniform ? 1 : v.size();
      for (size_t i = 0; i < n; i++) { snprintf(buf, sizeof buf, "%.17g", v[i]); out << (i ? "," : "") << buf; }
      out << "]";
    }
    out << "}";
  }
};

int main() {
  std::unique_ptr<Program> prog;
  std::map<long, Term::Ptr> T;
  std::unordered_map<std::string, std::string> cfg;
  std::map<std::string, std::vector<double>> evalInputs;
  bool evaluate = false;   // print reference_outputs (also for a program without inputs)
  std::string line;
  uint32_t scale = 0, range = 0;
  while (std::getline(std::cin, line)) {
    std::istringstream is(line);
    std::string cmd;
    if (!(is >> cmd) || cmd[0] == '#') continue;
    if (cmd == "program") { std::string name; uint64_t vs; is >> name >> vs; prog = std::make_unique<Program>(name, vs); }
    else if (cmd == "input") { long id; std::string name, ty; is >> id >> name >> ty;
      T[id] = prog->makeInput(name, ty == "raw" ? Type::Raw : ty == "plain" ? Type::Plain : Type::Cipher); }
    else if (cmd == "uconst") { long id; double v; is >> id >> v; T[id] = prog->makeUniformConstant(v); }
    else if (cmd == "dconst") { long id; size_t n; is >> id >> n; std::vector<double> v(n); for (auto &x : v) is >> x; T[id] = prog->makeDenseConstant(v); }
    else if (cmd == "term") { long id; std::string op; is >> id >> op; std::vector<Term::Ptr> a; long x; while (is >> x) a.push_back(T.at(x));
      Op o = op == "Add" ? Op::Add : op == "Sub" ? Op::Sub : op == "Mul" ? Op::Mul : op == "Negate" ? Op::Negate : Op::Undef;
      T[id] = prog->makeTerm(o, a); }
    else if (cmd == "rotl") { long id, a; int s; is >> id >> a >> s; T[id] = prog->makeLeftRotation(T.at(a), s); }
    else if (cmd == "rotr") { long id, a; int s; is >> id >> a >> s; T[id] = prog->makeRightRotation(T.at(a), s); }
    else if (cmd == "output") { std::string name; long a; is >> name >> a; prog->makeOutput(name, T.at(a)); }
    else if (cmd == "scales") is >> scale;
    else if (cmd == "ranges") is >> range;
    else if (cmd == "config") { std::string k, v; is >> k >> v; cfg[k] = v; }
    else if (cmd == "evaluate") evaluate = true;
    else if (cmd == "evalinput") { std::string name; size_t n; is >> name >> n; std::vector<double> v(n); for (auto &x : v) is >> x; evalInputs[name] = v; }
  }
  // what python/eva/wrapper.cpp:48-68 set_output_ranges / set_input_scales do
  for (auto &e : prog->getOutputs()) e.second->set<RangeAttribute>(range);
  for (auto &s : prog->getSources()) s->set<EncodeAtScaleAttribute>(scale);
  try {
    CKKSCompiler compiler{CKKSConfig(cfg)};
    auto res = compiler.compile(*prog);
    auto &cp = *std::get<0>(res);
    auto &params = std::get<1>(res);
    auto &sig = std::get<2>(res);
    std::cout << "{\"name\":" << jstr(cp.getName()) << ",\"vec_size\":" << cp.getVecSize() << ",\n";
    std::cout << "\"poly_modulus_degree\":" << params.polyModulusDegree << ",\"prime_bits\":[";
    for (size_t i = 0; i < params.primeBits.size(); i++) std::cout << (i ? "," : "") << params.primeBits[i];
    std::cout << "],\"rotations\":[";
    { bool f = true; for (int r : params.rotations) { std::cout << (f ? "" : ",") << r; f = false; } }
    std::cout << "],\n\"signature\":{";
    { std::map<std::string, CKKSEncodingInfo> ord(sig.inputs.begin(), sig.inputs.end()); bool f = true;
      for (auto &e : ord) { std::cout << (f ? "" : ",") << jstr(e.first) << ":{\"type\":" << jstr(getTypeName(e.second.inputType))
                                      << ",\"scale\":" << e.second.scale << ",\"level\":" << e.second.level << "}"; f = false; } }
    std::cout << "},\n\"inputs\":{";
    { std::map<std::string, Term::Ptr> ord(cp.getInputs().begin(), cp.getInputs().end()); bool f = true;
      for (auto &e : ord) { std::cout << (f ? "" : ",") << jstr(e.first) << ":" << e.second->index; f = false; } }
    std::cout << "},\"outputs\":{";
    { std::map<std::string, Term::Ptr> ord(cp.getOutputs().begin(), cp.getOutputs().end()); bool f = true;
      for (auto &e : ord) { std::cout << (f ? "" : ",") << jstr(e.first) << ":" << e.second->index; f = false; } }
    std::cout << "},\n\"terms\":[\n";
    Dumper d(cp);
    ProgramTraversal(cp).forwardPass(d);
    std::cout << d.out.str() << "\n]";
    if (evaluate || !evalInputs.empty()) {  // reference (plaintext) semantics: eva/eva.cpp:11-21
      Valuation in;
      for (auto &e : evalInputs) in[e.first] = e.second;
      ReferenceExecutor ex(cp);
      ex.setInputs(in);
      ProgramTraversal(cp).forwardPass(ex);
      Valuation outv;
      ex.getOutputs(outv);
      std::map<std::string, std::vector<double>> ord(outv.begin(), outv.end());
      std::cout << ",\n\"reference_outputs\":{";
      bool f = true; char buf[64];
      for (auto &e : ord) {
        std::cout << (f ? "" : ",") << jstr(e.first) << ":["; f = false;
        for (size_t i = 0; i < e.second.size(); i++) { snprintf(buf, sizeof buf, "%.17g", e.second[i]); std::cout << (i ? "," : "") << buf; }
        std::cout << "]";
      }
      std::cout << "}";
    }
    std::cout << "}\n";
  } catch (const std::exception &e) {
    std::cout << "{\"error\":" << jstr(e.what()) << "}\n";
  }
  return 0;
}
