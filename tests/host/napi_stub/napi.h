// napi.h — a stand-in for the subset of node-addon-api that integration/napi/snarkb200_napi.cc uses.  TEST INFRASTRUCTURE:
// there is no Node.js (and no node-addon-api) in this image or on the GPU box, so the shim cannot be built for its real
// host.  This header gives the same class and method names a small in-process implementation (values are tagged C++
// objects, an AsyncWorker runs Execute() and its completion callback synchronously inside Queue()), so that the shim
// compiles against the declared signatures, links against the real libsnarkb200.so and can be driven by
// tests/host/napi_shim_check.cpp.  It proves the C-ABI calls of the shim are well-typed and behave; it says nothing
// about N-API itself.
#pragma once
#include <cstdint>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace Napi {

struct Data {                       // one JS value
    enum Kind { Undefined, Number, String, Bytes, External, Object, Function, Error } kind = Undefined;
    double num = 0; std::string str; std::vector<uint8_t> bytes; void* ext = nullptr; std::function<void()> finalizer;
    std::map<std::string, std::shared_ptr<Data>> props;
    std::function<struct Value(const struct CallbackInfo&)> fn;
    ~Data() { if (finalizer) finalizer(); }
};
struct Env { Env() {} struct Value Undefined() const; };

struct Value {
    std::shared_ptr<Data> d;
    Value() : d(std::make_shared<Data>()) {}
    explicit Value(std::shared_ptr<Data> p) : d(std::move(p)) {}
    template <class T> T As() const { T t; t.d = d; return t; }
    Napi::Env Env() const { return Napi::Env(); }
};
inline Value Env::Undefined() const { return Value(); }

struct Number : Value {
    int32_t Int32Value() const { return (int32_t)d->num; }
    uint32_t Uint32Value() const { return (uint32_t)d->num; }
    int64_t Int64Value() const { return (int64_t)d->num; }
    static Number New(Napi::Env, double v) { Number n; n.d->kind = Data::Number; n.d->num = v; return n; }
};
struct String : Value {
    std::string Utf8Value() const { return d->str; }
    static String New(Napi::Env, const std::string& s) { String v; v.d->kind = Data::String; v.d->str = s; return v; }
};
struct Uint8Array : Value {
    size_t ByteLength() const { return d->bytes.size(); }
    uint8_t* Data() const { return d->bytes.data(); }
    static Uint8Array New(Napi::Env, const uint8_t* p, size_t n) { Uint8Array a; a.d->kind = Data::Bytes; a.d->bytes.assign(p, p + n); return a; }
};
template <class T> struct Buffer : Uint8Array {
    static Buffer Copy(Napi::Env, const T* p, size_t n) { Buffer b; b.d->kind = Napi::Data::Bytes; b.d->bytes.assign((const uint8_t*)p, (const uint8_t*)p + n * sizeof(T)); return b; }
};
template <class T> struct External : Value {
    T* Data() const { return (T*)d->ext; }
    template <class Fin> static External New(Napi::Env env, T* p, Fin fin) { External e; e.d->kind = Napi::Data::External; e.d->ext = p; e.d->finalizer = [env, p, fin]() { fin(env, p); }; return e; }
};
struct Object : Value {
    static Object New(Napi::Env) { Object o; o.d->kind = Data::Object; return o; }
    void Set(const char* k, const Value& v) { d->props[k] = v.d; }
    void Set(const char* k, uint32_t v) { d->props[k] = Number::New(Napi::Env(), v).d; }
    Value Get(const char* k) const { auto it = d->props.find(k); return it == d->props.end() ? Value() : Value(it->second); }
};
struct CallbackInfo {
    std::vector<Value> args;
    Napi::Env Env() const { return Napi::Env(); }
    Value operator[](size_t i) const { return i < args.size() ? args[i] : Value(); }
};
struct Function : Value {
    static Function New(Napi::Env, Value (*f)(const CallbackInfo&)) { Function v; v.d->kind = Data::Function; v.d->fn = f; return v; }
    Value Call(const std::vector<Value>& a) const { CallbackInfo ci; ci.args = a; return d->fn(ci); }
};
struct Error : Value {
    std::string Message() const { return d->str; }
    Value Value_() const { return *this; }
    Napi::Value Value() const { return *this; }
    static Error New(Napi::Env, const std::string& m) { Error e; e.d->kind = Data::Error; e.d->str = m; return e; }
    void ThrowAsJavaScriptException() const { pending() = d->str; }
    static std::string& pending() { static std::string p; return p; }     // the "exception" a synchronous binding left behind
};
template <class T> struct Reference { T v; };
template <class T> Reference<T> Persistent(T v) { return Reference<T>{v}; }

struct Promise : Value {
    struct Deferred {
        std::shared_ptr<Data> state = std::make_shared<Data>();     // props: "value" or "error"
        static Deferred New(Napi::Env) { return Deferred(); }
        void Resolve(const Value& v) { state->props["value"] = v.d; }
        void Reject(const Value& v) { state->props["error"] = v.d; }
        Napi::Promise Promise() const { Napi::Promise p; p.d = state; return p; }
    };
};
class AsyncWorker {
 public:
    explicit AsyncWorker(Napi::Env) {}
    virtual ~AsyncWorker() {}
    Napi::Env Env() const { return Napi::Env(); }
    void SetError(const std::string& m) { err_ = m; failed_ = true; }
    // Execute() and the completion callback run at once, but the worker is only deleted at exit: node-addon-api deletes it
    // after the completion callback, on a later turn of the event loop, so a binding may still read it after Queue().
    void Queue() { Execute(); if (failed_) OnError(Error::New(Env(), err_)); else OnOK(); completed().emplace_back(this); }
 protected:
    virtual void Execute() = 0;
    virtual void OnOK() {}
    virtual void OnError(const Error&) {}
 private:
    static std::vector<std::unique_ptr<AsyncWorker>>& completed() { static std::vector<std::unique_ptr<AsyncWorker>> w; return w; }
    std::string err_; bool failed_ = false;
};
}  // namespace Napi

// the module's Init is reachable by the driver through this symbol
#define NODE_API_MODULE(name, init) extern "C" Napi::Object napi_stub_init() { return init(Napi::Env(), Napi::Object::New(Napi::Env())); }
